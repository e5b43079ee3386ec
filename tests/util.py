import os

import numpy as np
import torch

from oracle import neuman_oracle as no
from oracle import scenes, synth_smpl

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def golden(name):
    return dict(np.load(os.path.join(GOLD, name)))


def pick(n, k, seed):
    """k seeded positions in [0, n) (all of them when n <= k), sorted: where a golden fixture samples a large array."""
    if n <= k:
        return np.arange(n)
    return np.sort(np.random.RandomState(seed).choice(n, k, replace=False))


def assert_state_dict_is_the_references(sd, G, prefix):
    """`sd` has the keys in the same order, the same shapes, and the same values: float64 sums and the
    values at the seeded positions the fixture `G` sampled (tools/make_golden_reference.py: state_digest)."""
    keys = [str(k) for k in G[f"{prefix}_keys"]]
    assert list(sd) == keys
    for i, k in enumerate(keys):
        v = sd[k].detach().cpu()
        assert "x".join(map(str, v.shape)) == str(G[f"{prefix}_shapes"][i]), k
        sums = np.array([v.double().sum().item(), v.double().abs().sum().item()])
        assert np.allclose(sums, G[f"{prefix}_sums"][i], rtol=1e-12, atol=1e-12), k
        idx = pick(v.numel(), G[f"{prefix}_vals"].shape[1], i)
        assert np.array_equal(v.reshape(-1)[torch.from_numpy(idx)].numpy(), G[f"{prefix}_vals"][i, :len(idx)]), k


def product_nets(device="cpu"):
    """(coarse, fine, human) seeded exactly like tools/make_golden.py."""
    import neuman_b200 as nb
    coarse, fine = scenes.seed_nets(nb.build_nerf, nb.default_opt(use_cuda=False), 1)
    human, _ = scenes.seed_nets(nb.build_nerf, nb.default_opt(use_cuda=False, posenc="rotate"), 2)
    return coarse.to(device), fine.to(device), human.to(device)


def product_human_model(device="cpu"):
    import neuman_b200 as nb
    torch.manual_seed(1)
    net = nb.HumanNeRF(nb.default_opt(use_cuda=False))
    scenes.boost_density(net.coarse_human_net)
    return net.to(device)


def oracle_params(joiner):
    return no.net_params_from_joiner(joiner)


def bodies():
    return (synth_smpl.random_body(seed=1, center=(0.1, 0.0, 0.3)),
            synth_smpl.random_body(seed=4, center=(-0.15, 0.0, 0.5)))


def psnr(a, b):
    mse = float(np.mean((np.asarray(a, dtype=np.float64) - np.asarray(b, dtype=np.float64)) ** 2))
    return 99.0 if mse == 0 else -10.0 * np.log10(mse)


# ---------------------------------------------------------------------------------------------
# Depth / colour gates with the measured 11-bit-operand floor (SURVEY.md §8d "noise floor next to every gate").
# north_star: <= 1e-4 abs against the reference path.  The default MLP mode multiplies fp16 operands (11 significand
# bits, like TF32); `floor16` is what that operand precision alone does to the ORACLE's own result on the same rays.  The
# tensor-core path is held to max(1e-4, K * floor16) with K = 1.5 (accumulation order, MUFU encodings); the fp32
# CUDA-core mode (NEUMAN_MLP_MODE=simt) to 1e-4.
# ---------------------------------------------------------------------------------------------
TOL = 1e-4
K_FLOOR = 1.5


def tc_mode():
    return os.environ.get("NEUMAN_MLP_MODE", "tc") != "simt"


def floors16(run):
    """run() -> tuple of numpy arrays (the oracle on some rays); returns max |fp32 - 11-bit operands| per output."""
    base = run()
    with no.precision(operands="f16"):
        tc = run()
    return [float(np.abs(np.asarray(a) - np.asarray(b)).max()) for a, b in zip(base, tc)]


def gate(err, floor16):
    """The bound for a maximum error `err` given the measured floor (see above)."""
    return max(TOL, K_FLOOR * floor16) if tc_mode() else TOL
