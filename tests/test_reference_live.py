"""The CUDA path and the oracle against the UNMODIFIED reference modules.

Numbers: against what the reference computed, recorded in ``tests/golden/reference_live.npz`` by
``tests/golden/make_golden_live.py`` (inputs and weights are regenerated from seeds; outputs too large to store whole are
kept as a fixed ``conftest.flat_sample`` plus their max-norm, which stays the denominator of the relative error).
CPU part (``-m "not gpu"``): the restatement oracle/spk_oracle.py against the reference, and -- where the reference's own
classes can be imported (oracle/ref_loader.py) -- ``convert_model`` on the reference's shipped trained model (class swap,
identical state_dict, fp64 -> fp32 cast).
GPU part: the CUDA path against the reference in fp64 at the FULL sizes of the named configurations (cfg2 B=256, cfg3
B=1024 padded, cfg4 8192 atoms), the block-level API (PaiNNInteraction / PaiNNMixing / SchNetInteraction forward +
gradients), and ``convert_model`` end to end (incl. custom nuclear / electronic embeddings) where the reference's classes
can be imported.
Tolerance: 1e-5 relative (max-norm) against fp64, BASELINE.json north_star.
"""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, flat_sample, rel_err

from oracle import ref_loader as rl

needs_ref = pytest.mark.skipif(not rl.available(), reason="the reference's own classes are not importable (oracle/ref_loader.py)")
TOL = 1e-5

# the recorded cases (tests/golden/make_golden_live.py evaluates the reference on exactly these)
ORACLE_CASES = (("cfg2", dict(batch=3)), ("cfg1", {}), ("cfg4", dict(n_atoms_total=200)))
ORACLE_SEED = 2
FULL_SIZE_SEED = 7
FORCES_SAMPLE = 4096
BLOCK_BATCH = dict(batch=4, seed=2)
BLOCK_SEED = 3
BLOCK_SAMPLE = 1024


def recorded():
    return np.load(os.path.join(GOLDEN, "reference_live.npz"))


def sampled_rel_err(got, z, key, k):
    """rel_err of ``got`` against the recorded ``flat_sample(ref, k)`` under ``key``, over the full reference's max-norm."""
    a = flat_sample(np.asarray(got, dtype=np.float64), k)
    return float(np.max(np.abs(a - z[key])) / max(float(z[key + ":max"]), 1e-30))


def block_cases(painn_interaction, painn_mixing, schnet_interaction, silu, ssp, batch, Fd=128):
    """(name, block, [(input shape, distribution)], call) of the block-level API, built from the given block classes:
    ``call(block, inputs, idx_i, idx_j)`` returns the list of the block's outputs."""
    N, E = batch["_atomic_numbers"].shape[0], batch["_idx_i"].shape[0]
    return [
        ("painn_interaction", painn_interaction(Fd, silu),
         [((N, 1, Fd), "normal"), ((N, 3, Fd), "normal"), ((E, 1, 3 * Fd), "normal"), ((E, 3), "normal")],
         lambda m, x, ii, jj: list(m(*x, ii, jj, N))),
        ("painn_mixing", painn_mixing(Fd, silu, 1e-8), [((N, 1, Fd), "normal"), ((N, 3, Fd), "normal")],
         lambda m, x, ii, jj: list(m(*x))),
        ("schnet_interaction", schnet_interaction(Fd, 20, Fd, ssp),
         [((N, Fd), "normal"), ((E, 20), "normal"), ((E,), "uniform")],
         lambda m, x, ii, jj: [m(x[0], x[1], ii, jj, x[2])]),
    ]


def block_draws(rng, block, inputs):
    """Seeded weights (xavier-uniform matrices, U(-0.1, 0.1) vectors) and inputs of one block case, drawn with numpy so
    that they are the same wherever they are drawn."""
    sd = {}
    for k, v in block.state_dict().items():
        a = np.sqrt(6.0 / sum(v.shape)) if v.dim() == 2 else 0.1
        sd[k] = torch.as_tensor(rng.uniform(-a, a, tuple(v.shape)).astype(np.float32))
    xs = [(rng.standard_normal(s) if d == "normal" else rng.uniform(0.0, 1.0, s)).astype(np.float32) for s, d in inputs]
    return sd, xs


# ------------------------------------------------------------------------------------------------------------ CPU
def test_oracle_matches_live_reference_cpu():
    from oracle import spk_oracle as O
    from schnetpack_b200 import synthetic as S

    z = recorded()
    for cfg, kw in ORACLE_CASES:
        spec, data = S.make_config(cfg, **kw)
        params = S.init_params(spec, seed=ORACLE_SEED)
        o = O.energy_forces(spec, params, data, dtype=torch.float64)
        assert rel_err(o["energy"].numpy(), z[f"oracle:{cfg}:energy"]) < 1e-12
        assert rel_err(o["forces"].numpy(), z[f"oracle:{cfg}:forces"]) < 1e-10


@needs_ref
def test_convert_model_swaps_classes_and_keeps_state_dict():
    """INTEGRATION.md section 1: convert_model(reference model) -> B200 modules with the SAME state_dict (keys and values),
    postprocessors reused, fp64 models cast to fp32 with input casting switched on."""
    import schnetpack_b200 as sb
    from schnetpack_b200 import atomistic, representation
    from schnetpack_b200.model import NeuralNetworkPotential, convert_model

    ref = rl.load_model(rl.testdata("md_ethanol.model"))
    new = convert_model(ref)
    assert isinstance(new, NeuralNetworkPotential) and isinstance(new.representation, representation.PaiNN)
    assert isinstance(new.input_modules[0], atomistic.PairwiseDistances)
    assert isinstance(new.output_modules[0], atomistic.Atomwise) and isinstance(new.output_modules[1], atomistic.Forces)
    assert [type(p).__name__ for p in new.postprocessors] == [type(p).__name__ for p in ref.postprocessors]
    sd0, sd1 = ref.state_dict(), new.state_dict()
    assert list(sd0) == list(sd1)
    for k in sd0:
        assert torch.equal(sd0[k], sd1[k]), k
    assert sorted(new.model_outputs) == sorted(ref.model_outputs)
    assert sorted(new.required_derivatives) == sorted(ref.required_derivatives)
    assert float(new.representation.cutoff) == float(ref.representation.cutoff)     # read by spkdeploy:38
    assert not new.training and not new.cast_inputs
    # fp64 model (spkmd loads every model as fp64 first, md/calculators/schnetpack_calculator.py:98)
    new64 = convert_model(rl.load_model(rl.testdata("md_ethanol.model")).double())
    assert all(p.dtype == torch.float32 for p in new64.parameters()) and new64.cast_inputs
    for k in sd0:
        assert torch.equal(sd0[k].float() if sd0[k].is_floating_point() else sd0[k], new64.state_dict()[k]), k


@needs_ref
def test_convert_model_accepts_shared_blocks_schnet_and_custom_embeddings():
    from schnetpack_b200.model import convert_model

    spk = rl.load()
    emb = spk.nn.embedding
    rep = spk.representation.PaiNN(64, 2, spk.nn.BesselRBF(16, 4.0), spk.nn.CosineCutoff(4.0), shared_interactions=True,
                                   shared_filters=True, nuclear_embedding=emb.NuclearEmbedding(101, 64, zero_init=False),
                                   electronic_embeddings=[emb.ElectronicEmbedding("total_charge", 64, is_charged=True)])
    model = spk.model.NeuralNetworkPotential(rep, input_modules=[spk.atomistic.PairwiseDistances()],
                                             output_modules=[spk.atomistic.Atomwise(n_in=64, output_key="energy"),
                                                             spk.atomistic.Forces()])
    new = convert_model(model)
    assert new.representation.interactions[0] is new.representation.interactions[1]
    assert new.representation.share_filters and type(new.representation.embedding).__name__ == "NuclearEmbedding"
    assert list(model.state_dict()) == list(new.state_dict())
    rep = spk.representation.SchNet(64, 3, spk.nn.GaussianRBF(20, 5.0), spk.nn.CosineCutoff(5.0), n_filters=64)
    model = spk.model.NeuralNetworkPotential(rep, input_modules=[spk.atomistic.PairwiseDistances()],
                                             output_modules=[spk.atomistic.Atomwise(n_in=64, output_key="energy")])
    assert list(model.state_dict()) == list(convert_model(model).state_dict())


# ------------------------------------------------------------------------------------------------------------ GPU
def _cuda_eval(model, data, dev):
    from schnetpack_b200.model import batch_to_device

    x = batch_to_device(data, dev)
    if "_Rij" in x:
        x = model.representation(x)
        x = model.output_modules[0](x)
        res = {"energy": x["energy"]}
    else:
        res = model(x)
    torch.cuda.synchronize()
    return {k: v.detach().cpu().numpy() for k, v in res.items()}


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", ["cfg2", "cfg3", "cfg4"])
def test_full_size_parity_against_reference_on_gpu(cfg):
    """The benchmarked sizes themselves: cfg2 = aspirin x 256 (5376 atoms / 78 k edges, PaiNN E+F), cfg3 = QM9-like x 1024
    with the padded neighbour list (831 488 edge slots, SchNet 128x6, energy), cfg4 = 8192-atom periodic box (PaiNN E+F).
    Checker: the reference's own modules in fp64."""
    from schnetpack_b200 import synthetic as S
    from schnetpack_b200.model import from_spec

    z = recorded()
    dev = torch.device("cuda:0")
    spec, data = S.make_config(cfg)
    params = S.init_params(spec, seed=FULL_SIZE_SEED)
    assert [data["_atomic_numbers"].shape[0], data["_idx_i"].shape[0]] == z[f"full:{cfg}:atoms_edges"].tolist()
    out = _cuda_eval(from_spec(spec, params, dev), data, dev)
    e = rel_err(out["energy"], z[f"full:{cfg}:energy"])
    print(cfg, "N", data["_atomic_numbers"].shape[0], "E", data["_idx_i"].shape[0], "energy rel err", e)
    assert e < TOL
    assert ("forces" in out) == (f"full:{cfg}:forces" in z.files)
    if "forces" in out:
        f = sampled_rel_err(out["forces"], z, f"full:{cfg}:forces", FORCES_SAMPLE)
        print(cfg, "forces rel err", f)
        assert f < TOL


@pytest.mark.gpu
@needs_ref
def test_convert_model_end_to_end_on_gpu():
    """convert_model(reference trained PaiNN) on the reference's own test geometry: energies / forces (postprocessors on:
    CastTo64 + AddOffsets) equal the reference's to 1e-5 -- and the fp64-loaded model path of spkmd too."""
    from schnetpack_b200 import synthetic as S
    from schnetpack_b200.model import batch_to_device, convert_model

    dev = torch.device("cuda:0")
    data = S.ethanol_batch(4, jitter=0.05, seed=3)
    ref = rl.load_model(rl.testdata("md_ethanol.model")).double().to(dev)
    want = ref({k: (v.double() if v.is_floating_point() else v) for k, v in batch_to_device(data, dev).items()})
    for dtype in (torch.float32, torch.float64):
        src = rl.load_model(rl.testdata("md_ethanol.model")).to(dtype)
        new = convert_model(src).to(dev)
        x = {k: (v.to(dtype) if v.is_floating_point() else v) for k, v in batch_to_device(data, dev).items()}
        got = new(x)
        assert got["forces"].dtype == (torch.float64 if dtype == torch.float64 else got["forces"].dtype)
        for k in ("energy", "forces"):
            err = rel_err(got[k].detach().cpu().numpy(), want[k].detach().cpu().numpy())
            print("convert_model", dtype, k, err)
            assert err < TOL, (dtype, k, err)


@pytest.mark.gpu
@needs_ref
def test_convert_model_custom_embeddings_on_gpu():
    """Models with NuclearEmbedding / ElectronicEmbedding (no ``.weight``; run as given) through convert_model."""
    from schnetpack_b200 import synthetic as S
    from schnetpack_b200.model import batch_to_device, convert_model

    dev = torch.device("cuda:0")
    spk = rl.load()
    emb = spk.nn.embedding
    torch.manual_seed(0)
    rep = spk.representation.PaiNN(128, 2, spk.nn.GaussianRBF(20, 5.0), spk.nn.CosineCutoff(5.0),
                                   nuclear_embedding=emb.NuclearEmbedding(101, 128, zero_init=False),
                                   electronic_embeddings=[emb.ElectronicEmbedding("total_charge", 128, is_charged=True)])
    model = spk.model.NeuralNetworkPotential(rep, input_modules=[spk.atomistic.PairwiseDistances()],
                                             output_modules=[spk.atomistic.Atomwise(n_in=128, output_key="energy"),
                                                             spk.atomistic.Forces()]).eval()
    data = S.aspirin_batch(5, seed=1)
    data["total_charge"] = np.array([0.0, 1.0, -1.0, 2.0, 0.0], dtype=np.float32)
    data["_idx"] = np.arange(5, dtype=np.int64)              # read by ElectronicEmbedding (nn/embedding.py:311)
    new = convert_model(model).to(dev)
    got = new(batch_to_device(data, dev))
    ref = model.double().to(dev)
    want = ref({k: (v.double() if v.is_floating_point() else v) for k, v in batch_to_device(data, dev).items()})
    for k in ("energy", "forces"):
        assert rel_err(got[k].detach().cpu().numpy(), want[k].detach().cpu().numpy()) < TOL, k


@pytest.mark.gpu
def test_block_level_api_matches_reference_blocks():
    """PaiNNInteraction.forward(q, mu, Wij, dir_ij, idx_i, idx_j, n_atoms), PaiNNMixing.forward(q, mu) and
    SchNetInteraction.forward(x, f_ij, idx_i, idx_j, rcut_ij) called directly, values and first-order gradients, against the
    reference's blocks with the same weights (fp64)."""
    import torch.nn.functional as F_

    from schnetpack_b200 import representation as R
    from schnetpack_b200 import synthetic as S
    from schnetpack_b200.nn import shifted_softplus

    z = recorded()
    dev = torch.device("cuda:0")
    b = S.aspirin_batch(**BLOCK_BATCH)
    ii, jj = torch.as_tensor(b["_idx_i"], device=dev), torch.as_tensor(b["_idx_j"], device=dev)
    rng = np.random.RandomState(BLOCK_SEED)
    tol = 5e-6
    for name, blk, inputs, call in block_cases(R.PaiNNInteraction, R.PaiNNMixing, R.SchNetInteraction, F_.silu,
                                               shifted_softplus, b):
        sd, xs = block_draws(rng, blk, inputs)
        blk.load_state_dict(sd)
        blk = blk.to(dev).eval()
        ins = [torch.as_tensor(x, device=dev).requires_grad_() for x in xs]
        outs = call(blk, ins, ii, jj)
        seeds = [torch.as_tensor(rng.standard_normal(tuple(o.shape)).astype(np.float32), device=dev) for o in outs]
        g = torch.autograd.grad(sum((o * s).sum() for o, s in zip(outs, seeds)), ins)
        for i, o in enumerate(outs):
            assert sampled_rel_err(o.detach().cpu().numpy(), z, f"block:{name}:out{i}", BLOCK_SAMPLE) < tol, (name, i)
        for i, a in enumerate(g):
            assert sampled_rel_err(a.cpu().numpy(), z, f"block:{name}:grad{i}", BLOCK_SAMPLE) < 2 * tol, (name, i)
