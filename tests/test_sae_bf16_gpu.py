"""cfg #5 shape class: a bfloat16 SAE (``_dtype="bfloat16"``) trained through VisionSAETrainer.train_step.

Storage is what the reference's would be (bf16 nn.Parameters / state dict / activations); the optimizer math, the Adam moments and
the accumulated parameters are fp32 masters inside the step engine (the reference keeps bf16 only).  The fixture
(tests/golden/make_golden_sae_bf16.py, unmodified reference + a one-entry dtype_mapping shim) holds two trajectories from the same
bf16 initial state: the reference in bf16 and the reference in fp32.  Bars:
  * step-0 reconstruction on identical bf16 weights: one bf16 rounding from the reference's fp32 output; its bf16 output is itself
    8e-2 from that (bf16 ties change the TopK support), so against it the bar is the triangle inequality, not 1e-2;
  * losses: within 1e-2 of the reference's bf16 run, within 1e-4 of its fp32 run (our arithmetic is the fp32 one);
  * parameters after every step: bf16 tensors, no further from the fp32 trajectory than one bf16 rounding (2^-8 relative); the two
    matrices never further from it than the reference's own bf16 run is (the biases are printed, not asserted: a parameter the
    reference's bf16 Adam happens not to move at all can sit closer to the fp32 run than one rounding).
"""
import contextlib
import io

import pytest
import torch

pytestmark = pytest.mark.gpu

from tests.util import load_golden, rel_err  # noqa: E402


def _trainer(gold):
    from vit_prisma.sae.config import VisionModelSAERunnerConfig
    from vit_prisma.sae.train_sae import VisionSAETrainer
    with contextlib.redirect_stdout(io.StringIO()):
        cfg = VisionModelSAERunnerConfig(d_in=gold["d_in"], expansion_factor=gold["d_sae"] // gold["d_in"], activation_fn_str="topk",
                                         activation_fn_kwargs={"k": gold["k"]}, _device="cuda", _dtype="bfloat16",
                                         normalize_activations=gold["norm"], b_dec_init_method="zeros", lr=gold["lr"],
                                         lr_warm_up_steps=gold["warm_up_steps"], train_batch_size=gold["batch"], max_grad_norm=1.0,
                                         initialization_method="independent", log_to_wandb=False, n_checkpoints=0,
                                         checkpoint_path="/tmp/prisma_b200_unused",
                                         # total_training_steps is derived: int(1.3e6 * num_epochs) images x context_size tokens // batch
                                         num_epochs=(gold["total_steps"] + 0.5) / 1_300_000, context_size=gold["batch"])
    assert cfg.total_training_steps == gold["total_steps"]
    trainer = VisionSAETrainer(cfg, model=None, dataset=None, activations_store=object())
    sae = trainer.sparse_coder
    sae.load_state_dict({k: v.cuda() for k, v in gold["init"].items()})
    return cfg, trainer, sae


def test_bf16_sae_trains_on_fp32_masters_and_exports_bf16_parameters():
    gold = load_golden("sae_bf16_v.pt")
    cfg, trainer, sae = _trainer(gold)
    assert all(v.dtype == torch.bfloat16 for v in sae.state_dict().values())
    data = gold["data"].cuda()
    B = gold["batch"]
    # step-0 reconstruction through the module's own forward (bf16 weights identical to the reference's)
    sae.eval()
    sae.set_decoder_norm_to_unit_norm()                          # the reference's loop normalises before its first forward (train_sae.py:306)
    out0 = sae(data[:B])[0]
    assert out0.dtype == torch.bfloat16
    e32 = rel_err(out0.float().cpu(), gold["steps_fp32"][0]["sae_out"])
    e16 = rel_err(out0.float().cpu(), gold["steps"][0]["sae_out"].float())
    r16 = rel_err(gold["steps"][0]["sae_out"].float(), gold["steps_fp32"][0]["sae_out"])
    print(f"step-0 sae_out: ours vs fp32 run {e32:.2e}, ours vs bf16 run {e16:.2e}, bf16 run vs fp32 run {r16:.2e}")
    assert e32 <= 2.0 ** -8          # fp32 arithmetic, one rounding of the output to bf16
    # The reference's OWN bf16 output is 8e-2 (max-norm) from its fp32 output on this fixture: hidden_pre rounded to bf16 ties and
    # reorders pre-activations near the k-th, so its TopK support differs from the exact one on some rows and whole features come
    # or go.  No implementation can be within 1e-2 of that output AND of the truth; the bars are therefore: one bf16 rounding from
    # the fp32 run (above), no further from the bf16 run than the bf16 run is from fp32 (triangle), closer to fp32 than it is.
    assert e16 <= r16 + e32 + 1e-3
    assert e32 <= r16 + 1e-3
    act_freq, since_fired, n_frac, opt, sched = trainer.initialize_training_variables()
    for s, (rec16, rec32) in enumerate(zip(gold["steps"], gold["steps_fp32"])):
        x = data[s * B:(s + 1) * B].unsqueeze(1)
        loss, mse, l1, l0, act_freq, since_fired, n_frac = trainer.train_step(sae, opt, sched, act_freq, since_fired, n_frac, x, s, s * B)
        assert abs(mse.item() - rec32["mse"]) <= 1e-4 * rec32["mse"], (s, mse.item(), rec32["mse"])
        assert abs(mse.item() - rec16["mse"]) <= 1e-2 * rec16["mse"], (s, mse.item(), rec16["mse"])
        assert abs(l0.item() - rec32["l0"]) < 1e-5
        sd = sae.state_dict()
        for name, ref32 in rec32["params_after"].items():
            mine = sd[name]
            assert mine.dtype == torch.bfloat16, name
            if name == "W_dec":                                   # the step leaves the rows unit-norm; the reference renormalises at its next step
                ref32 = ref32 / ref32.norm(dim=1, keepdim=True)
                ref16 = rec16["params_after"][name].float()
                ref16 = ref16 / ref16.norm(dim=1, keepdim=True)
            else:
                ref16 = rec16["params_after"][name].float()
            scale = float(ref32.abs().max())
            ours = float((mine.float().cpu() - ref32).abs().max())
            theirs = float((ref16 - ref32).abs().max())
            # one bf16 rounding of the fp32 trajectory: |x - bf16(x)| <= 2^-8 |x| (half a spacing relative to the bottom of a binade)
            assert ours <= 1.01 * 2.0 ** -8 * scale + 1e-7, f"step {s} {name}: {ours:.3e} from the fp32 trajectory (one bf16 rounding = {2.0 ** -8 * scale:.3e})"
            print(f"step {s} {name}: ours {ours:.2e} / reference-bf16 {theirs:.2e} from the fp32 trajectory (scale {scale:.2e})")
            if name in ("W_dec", "W_enc"):     # the matrices: the reference's bf16 Adam drifts by several roundings (2e-3 .. 6e-3 on W_dec, generator log)
                assert ours <= theirs + 2.0 ** -9 * scale + 1e-7, f"step {s} {name}: further from the fp32 trajectory ({ours:.3e}) than the reference's bf16 run ({theirs:.3e})"
    # the masters follow a load_state_dict (version check), and the module forward sees the trained parameters
    eng = sae.step_engine()
    assert eng.W_dec.dtype == torch.float32 and eng.m_dec.dtype == torch.float32
    assert rel_err(sae.W_dec.data.float(), eng.W_dec) <= 2.0 ** -8
    sae.load_state_dict({k: v.cuda() for k, v in gold["init"].items()})
    eng2 = sae.step_engine()
    assert torch.equal(eng2.W_dec.cpu(), gold["init"]["W_dec"].float())


def test_bf16_module_routes_agree_and_hooks_see_bf16():
    """A bf16 module computes in fp32 on its masters on BOTH routes: the sparse engine route (no hooks) and the module-by-module route
    (a HookPoint is live).  Hooks see tensors rounded to cfg.dtype -- the reference's rounding points -- and the two routes agree to
    bf16 rounding; encode / decode return cfg.dtype like the reference's do."""
    gold = load_golden("sae_bf16_v.pt")
    cfg, trainer, sae = _trainer(gold)
    sae.eval()
    x = gold["data"][:gold["batch"]].cuda()
    out_sparse = sae(x)
    seen = {}
    def grab(t, hook):
        seen[hook.name] = (t.dtype, tuple(t.shape))
        return None
    out_hooked = sae.run_with_hooks(x, fwd_hooks=[("hook_hidden_pre", grab), ("hook_sae_out", grab)])
    assert seen["hook_hidden_pre"] == (torch.bfloat16, (gold["batch"], gold["d_sae"]))
    assert seen["hook_sae_out"][0] == torch.bfloat16
    assert out_hooked[0].dtype == torch.bfloat16 and out_sparse[0].dtype == torch.bfloat16
    # the hooked route rounds hidden_pre to bf16 before TopK (as the reference does): bf16 ties change the support on some rows, which
    # is what puts the reference's own bf16 output 8e-2 from its fp32 output on this fixture -- same order of magnitude expected here
    assert rel_err(out_hooked[0].float(), out_sparse[0].float()) <= 1e-1
    assert abs(out_hooked[3].item() - out_sparse[3].item()) <= 5e-2 * abs(out_sparse[3].item())
    sae_in, feats = sae.encode(x)
    assert sae_in.dtype == torch.bfloat16 and feats.dtype == torch.bfloat16 and feats.shape == (gold["batch"], gold["d_sae"])
    assert int((feats > 0).sum(dim=1).max()) <= gold["k"]
    assert sae.decode(feats).dtype == torch.bfloat16
