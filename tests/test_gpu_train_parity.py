"""-m gpu: end-to-end TRAIN-mode parity of one IRFD generator step (train.py:186-203, differentiable losses) against
the CPU oracle, every gradient tensor compared — the check that pins backward ROUTING (which tensor feeds which kernel),
not just each kernel on its own inputs — plus style mixing against the oracle with truncation live (ADVICE r1 high).

Bounds are <= 2x the values measured on B200 (printed by `pytest -m gpu -s`; table in DESIGN.md §5).
"""
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

pytestmark = pytest.mark.gpu


def test_conditioned_train_step_all_gradients(cuda_device):
    """Oracle (CPU fp32, reentrant checkpoints) vs product (bf16 tensor-core path), identical conditioned weights
    (bn3 gamma x 0.2), inputs, swap draw and noise planes; style mixing off (its latent comes from the device RNG).
    Compares both losses, the six feature codes, both images, ALL 560 gradient tensors and ALL BN buffers."""
    import irfd_oracle as O
    from parity_util import conditioned_pair, g_step_oracle, g_step_product, grad_report

    dev = cuda_device
    ref, prod = conditioned_pair(dev, bn3_scale=0.2)
    x_s, x_t = O.synthetic_pair(2)
    r = g_step_oracle(ref, x_s, x_t, noise_seed=41, device="cpu")
    p = g_step_product(prod, x_s, x_t, noise_seed=41, device=dev)
    print("[parity] conditioned (bn3 gamma x 0.2) G train step, product vs CPU oracle, 2 pairs @256^2")
    rep = grad_report(r, p, verbose=True)
    assert rep["same_grad_set"] and len(r["grads"]) == 560
    assert rep["counters_equal"]                      # num_batches_tracked == 4 everywhere (SURVEY Q3)
    assert rep["running_mean"] < BOUNDS["running_mean"] and rep["running_var"] < BOUNDS["running_var"]
    assert rep["feat"] < BOUNDS["feat"] and rep["img"] < BOUNDS["img"]
    assert rep["loss_id"] < BOUNDS["loss_id"] and rep["loss_rec"] < BOUNDS["loss_rec"]
    for k, v in rep.items():
        if isinstance(v, tuple):
            med_b, worst_b = BOUNDS[k.split(".", 1)[1] if k[:2] in ("Ei", "Ee", "Ep") else k]
            assert v[0] < med_b and v[1] < worst_b, (k, v)


def test_train_step_vs_bf16_faithful_oracle(cuda_device):
    """The routing check proper: the oracle with the product's storage rounding points inserted (parity_util.
    make_bf16_faithful) on the conditioned weights (bn3 gamma x 0.2), one G train step.  With the same rounding points
    the ReLU masks agree, so every one of the 560 gradient tensors is compared at a bound a mis-routed tensor cannot
    meet.  (Without the conditioning even this oracle drifts: scripts/faithful_probe.py shows the 1.7e-5 difference the
    fp32 accumulation order leaves after the stem conv growing ~1.3x per layer to 0.3 in layer4 — the random-init
    train-mode stack is chaotic at that depth, SURVEY §7.)"""
    import irfd_oracle as O
    from parity_util import conditioned_pair, g_step_oracle, g_step_product, grad_report, make_bf16_faithful

    dev = cuda_device
    ref, prod = conditioned_pair(dev, bn3_scale=0.2)
    make_bf16_faithful(ref)
    x_s, x_t = O.synthetic_pair(2)
    r = g_step_oracle(ref, x_s, x_t, noise_seed=43, device="cpu")
    p = g_step_product(prod, x_s, x_t, noise_seed=43, device=dev)
    print("[parity] G train step, product vs bf16-faithful CPU oracle (same rounding points), 2 pairs @256^2")
    rep = grad_report(r, p, verbose=True)
    assert rep["same_grad_set"] and rep["counters_equal"]
    assert rep["feat"] < FAITHFUL["feat"] and rep["img"] < FAITHFUL["img"]
    assert rep["loss_id"] < FAITHFUL["loss"] and rep["loss_rec"] < FAITHFUL["loss"]
    assert rep["running_mean"] < FAITHFUL["running"] and rep["running_var"] < FAITHFUL["running"]
    for k, v in rep.items():
        if isinstance(v, tuple):
            med_b, worst_b = FAITHFUL[k if k.startswith("Gd") else "enc"]
            assert v[0] < med_b and v[1] < worst_b, (k, v)


# <= 2x measured on B200: features 3.7e-3, images 7.8e-3, l_identity 4.9e-5, l_recon 1.3e-3, running buffers 2.2e-3;
# Gd.synthesis 4.1e-3 / 3.7e-2, Gd.mapping 3.9e-2 / 5.2e-2, Gd.noise 5.0e-2 / 6.7e-2 (median / worst).
# Encoder gradients: median 0.25 (layer4) .. 0.35 (layer1), worst 0.56.  Forward and generator agree 2-3x better than
# with the pure-fp32 oracle, the encoder gradients do not: scripts/numerics_probe_cpu.py shows on the oracle alone that
# bf16 storage of the forward activations moves these gradients by 0.30-0.35 (ReLU-mask flips; rounding only the
# gradients costs 4e-3), and two implementations that agree to 4e-3 in the forward do not flip the SAME elements.  The
# encoder bound therefore only catches a gross mis-routing (uncorrelated gradients sit at 1.4); the sharp routing checks
# of the encoder backward are test_encoder_backward_eval_end_to_end (eval-mode BN, every gradient, median 2.5e-2),
# test_gpu_encoder_single.py::test_train_backward_in_context (every train-mode launch on its own inputs) and
# test_encoder_group_train_equals_three_passes (three-encoder lockstep pass against three one-encoder passes).
FAITHFUL = {"feat": 8e-3, "img": 1.6e-2, "loss": 3e-3, "running": 5e-3,
            "Gd.synthesis": (1e-2, 8e-2), "Gd.mapping": (8e-2, 0.11), "Gd.noise": (0.1, 0.14), "enc": (0.7, 1.1)}


# (median, worst) rel-L2 bounds per gradient group; scalars for the rest.  All <= 2x the values measured on B200:
# features 6.0e-3, images 1.2e-2, l_identity 1.2e-3, l_recon 2.8e-3, running mean/var 4.1e-3 / 3.5e-3,
# Gd.mapping 4.9e-2 / 6.6e-2, Gd.synthesis 1.3e-2 / 4.1e-2, Gd.noise 5.9e-2 / 1.2e-1.
# Encoder gradients against the PURE-fp32 oracle: median 0.32 (layer4) .. 0.50 (stem), worst 0.69 — flat over depth
# and the same for bn3 gamma x 0.05 (0.24 .. 0.32): it is not compounding rounding but the ReLU-mask flips of a bf16
# forward (see parity_util.make_bf16_faithful); test_train_step_vs_bf16_faithful_oracle is the sharp check.
BOUNDS = {
    "feat": 1.2e-2, "img": 2.4e-2, "loss_id": 3e-3, "loss_rec": 6e-3, "running_mean": 8e-3, "running_var": 7e-3,
    "Gd.mapping": (0.1, 0.13), "Gd.synthesis": (2.7e-2, 8e-2), "Gd.noise": (0.12, 0.24),
    "stem": (1.0, 1.1), "layer1": (0.95, 1.3), "layer2": (0.93, 1.1), "layer3": (0.85, 1.0), "layer4": (0.66, 0.83),
}


def _mixing_seeds():
    """Seeds whose CPU draws give: mixing with a cut below the truncation cutoff (the case ADVICE r1 found wrong),
    mixing with a cut at/above it, and no mixing."""
    want = {"low": None, "high": None, "none": None}
    for s in range(200):
        torch.manual_seed(s)
        r = float(torch.rand(1))
        if r < 0.9:
            cut = int(torch.randint(1, 14, (1,)))
            key = "low" if cut < 8 else "high"
        else:
            cut, key = 14, "none"
        if want[key] is None:
            want[key] = (s, cut)
        if all(v is not None for v in want.values()):
            break
    return want


def test_style_mixing_matches_oracle_eager_and_static(cuda_device):
    """StyleGenerator in train mode with style mixing ON: the oracle's Gd runs in fp32 on the same device, so both
    sides consume the CPU generator (rand, randint) and the device generator (randn_like) identically.  Rows below the
    cut are truncated (psi 0.7 for rows < 8), rows from the cut on are w2's UNtruncated rows (styleganv1.py:536-553)."""
    import irfd_oracle as O
    import speak_hack_b200 as P
    from parity_util import oracle_noise, product_noise

    dev = cuda_device
    torch.manual_seed(O.WEIGHT_SEED)
    ref = O.StyleGeneratorRef(input_dim=6144)
    O.perturb_noise_weights(ref)
    prod = P.StyleGenerator(input_dim=6144)
    prod.load_state_dict(ref.state_dict())
    ref, prod = ref.to(dev).train(), prod.to(dev).train()
    feat = (torch.randn(2, 6144, generator=torch.Generator().manual_seed(3)).abs() * 0.5).to(dev)
    L = prod.synthesis.num_layers
    for key, (seed, cut) in _mixing_seeds().items():
        oracle_noise(ref, 50 + seed)
        torch.manual_seed(seed)
        with torch.no_grad():
            rows_ref = ref.rows(feat)
        torch.manual_seed(seed)
        with torch.no_grad():
            img_ref = ref(feat)
        # eager product
        product_noise(prod, 50 + seed)
        torch.manual_seed(seed)
        with torch.no_grad():
            img = prod(feat)
        # static-graph flavour: the cut arrives through the control tensor, w2 is always drawn
        product_noise(prod, 50 + seed)
        ctrl = torch.tensor([0, cut, L], dtype=torch.int32, device=dev)
        torch.manual_seed(seed)
        with torch.no_grad():
            img_st = prod.forward_static(feat, ctrl, 1)
        torch.cuda.synchronize()
        e, e_st = O.rel_l2(img, img_ref), O.rel_l2(img_st, img_ref)
        # what the round-1 bug produced: truncated w2 rows in [cut, 8)
        trunc_w2 = rows_ref.clone()
        trunc_w2[:, cut:8] *= 0.7
        print(f"[parity] style mixing '{key}' (seed {seed}, cut {cut}): eager {e:.3e}, static {e_st:.3e} "
              f"(rows differ from the truncated-w2 variant by {O.rel_l2(trunc_w2, rows_ref):.3e})")
        assert torch.equal(img, img_st)      # same kernels, same rows: the two entry points must agree bit for bit
        assert e < 2.5e-2, (key, e)          # generator alone, bf16 path (measured ~1e-2)
