"""GPU: batched attack drivers (SURVEY 8f rank 1) against the reference's OWN attack classes -- `APGDAttack` and `FGSM` of
src/attacks/untargeted.py, imported unmodified through oracle/ref_import.py (skipped where that tree is absent) and run one image at a
time, as src/experiments/test_defense.py does -- on the same network, start noise and labels."""
import pytest
import torch

from gen_adversarial_b200 import ops, synth
from gen_adversarial_b200.attacks import APGDL2, FGSML2, dlr_loss
from oracle import ref_import

pytestmark = pytest.mark.gpu
needs_reference = pytest.mark.skipif(not ref_import.reference_available(), reason="reference tree not found (oracle/ref_import.py)")
DEV = "cuda:0"


def _ref_attacks():
    ref_import.install()
    import importlib
    return importlib.import_module("src.attacks.untargeted")


class _SmallNet(torch.nn.Module):
    def __init__(self, n_classes=10):
        super().__init__()
        g = torch.Generator().manual_seed(0)
        self.c1 = torch.nn.Conv2d(3, 16, 3, padding=1)
        self.c2 = torch.nn.Conv2d(16, 32, 3, padding=1)
        self.fc = torch.nn.Linear(32 * 8 * 8, n_classes)
        for p in self.parameters():
            p.data = torch.randn(p.shape, generator=g) * (0.3 if p.dim() > 1 else 0.05)

    def forward(self, x):
        x = torch.nn.functional.avg_pool2d(torch.tanh(self.c1(x)), 2)
        x = torch.nn.functional.avg_pool2d(torch.tanh(self.c2(x)), 2)
        return self.fc(x.flatten(1))


def test_apgd_step_kernel_matches_reference_update():
    g = torch.Generator().manual_seed(1)
    x = torch.rand(5, 3, 32, 32, generator=g)
    x_adv = (x + 0.05 * torch.randn(x.shape, generator=g)).clamp(0, 1)
    x_old = (x + 0.05 * torch.randn(x.shape, generator=g)).clamp(0, 1)
    grad = torch.randn(x.shape, generator=g)
    steps = torch.rand(5, generator=g) + 0.1
    bound, a = 0.7, 0.75
    rows = []
    for i in range(5):                                         # untargeted.py:176-193, one image at a time
        img, xa, xo, gr = x[i:i + 1], x_adv[i:i + 1], x_old[i:i + 1], grad[i:i + 1]
        nrm = lambda t: (t ** 2).sum().sqrt()
        grad2 = xa - xo
        new = xa + steps[i] * gr / nrm(gr)
        new = (new - img) / nrm(new - img) * torch.minimum(torch.tensor(bound), nrm(new - img))
        new = (img + new).clamp(0, 1)
        new = xa + (new - xa) * a + grad2 * (1 - a)
        new = (new - img) / nrm(new - img) * torch.minimum(torch.tensor(bound), nrm(new - img))
        rows.append((img + new).clamp(0, 1))
    ref = torch.cat(rows)
    xa_d, xo_d = x_adv.to(DEV).clone(), x_old.to(DEV).clone()
    ops.apgd_l2_step_(xa_d, xo_d, grad.to(DEV), x.to(DEV), steps.to(DEV), a, bound)
    assert (xa_d.cpu() - ref).abs().max().item() <= 2e-6
    assert torch.equal(xo_d.cpu(), x_adv)
    # FGSM step and the APGD starting point
    sg = torch.sign(grad)
    ref_f = (x + 0.5 * sg / sg.flatten(1).norm(dim=1).view(-1, 1, 1, 1)).clamp(0, 1)
    assert (ops.fgsm_l2_step(x.to(DEV), grad.to(DEV), 0.5).cpu() - ref_f).abs().max().item() <= 1e-6
    ref_s = (x + bound * grad / grad.flatten(1).norm(dim=1).view(-1, 1, 1, 1)).clamp(0, 1)
    assert (ops.l2_ball_start(x.to(DEV), grad.to(DEV), bound).cpu() - ref_s).abs().max().item() <= 1e-6


@needs_reference
@pytest.mark.parametrize("ce", [True, False])
def test_batched_apgd_matches_reference_class(ce, monkeypatch):
    ua = _ref_attacks()
    net = _SmallNet().to(DEV).eval()
    g = torch.Generator().manual_seed(2)
    b = 6
    x = torch.rand(b, 3, 32, 32, generator=g).to(DEV)
    noise = torch.randn(b, 3, 32, 32, generator=g).to(DEV)
    with torch.no_grad():
        y = net(x).argmax(1)
    n_iter, rho, bound = 25, 0.75, 0.8
    succ, l2, adv = APGDL2(n_iter, rho, bound, ce_loss=ce)(x, y, net, initial_noise=noise)
    ref_attack = ua.APGDAttack(n_iter, rho, bound, ce)
    same = 0
    for i in range(b):
        monkeypatch.setattr(torch, "randn_like", lambda t, _n=noise[i:i + 1]: _n.clone())
        s_ref, b_ref, adv_ref = ref_attack(x[i:i + 1], y[i:i + 1], net)
        monkeypatch.undo()
        d = (adv[i:i + 1] - adv_ref).abs().max().item()
        print(f"APGD-{'CE' if ce else 'DLR'} image {i}: success {bool(succ[i])} / ref {s_ref}, l2 {l2[i].item():.5f} / ref {b_ref:.5f}, max |adv - ref| {d:.2e}")
        assert bool(succ[i]) == bool(s_ref)
        assert abs(l2[i].item() - b_ref) <= 1e-3
        same += int(d <= 1e-4)
        assert l2[i].item() <= bound + 1e-4
    # the iteration has discrete decisions (loss > best, step halving): a near-tie can send one image down another branch
    assert same >= b - 1


@needs_reference
def test_batched_fgsm_matches_reference_class_on_the_defense():
    """FGSML2 on a whole batch through the fused loss_input_grad primitive against the reference's FGSM class driving the SAME defense
    model one image at a time through torch autograd (untargeted.py:708-750); fixed Philox seed, per-image sample offsets."""
    ua = _ref_attacks()
    from gen_adversarial_b200.nvae_spec import NvaeSpec, tiny_config
    from gen_adversarial_b200.defenses.ours.models import NVAEDefenseModel, CelebaIdentityClassifier
    cfg, res = tiny_config(initial_channels=16, groups=2, scales=2, latent=4), (3, 32, 32)
    spec = NvaeSpec(cfg, res)
    clf = CelebaIdentityClassifier({"state_dict": synth.make_vgg11_state_dict(10, seed=3, device=DEV)}, DEV, mode="fp32", n_classes=10, image_size=32)
    dm = NVAEDefenseModel(clf, synth.make_nvae_checkpoint(cfg, res, seed=3), [0.3] * spec.n_latents, 1.0, 0.5, True, DEV, mode="fp32").eval()
    dm.noise_seed = 11
    b = 5
    x = synth.synthetic_batch(b, res, 10, seed=4)[0].to(DEV)
    with torch.no_grad():
        y = dm(x).argmax(1)
    y[0] = (y[0] + 1) % 10                                       # one image the network already "misclassifies"
    succ, l2, adv = FGSML2(1.5)(x, y, dm)
    ref_attack = ua.FGSM(1.5)
    for i in range(b):
        dm.sample_offset = i                                      # the batch-1 call must draw image i's noise stream
        s_ref, b_ref, adv_ref = ref_attack(x[i:i + 1], y[i:i + 1], dm)
        dm.sample_offset = 0
        assert bool(succ[i]) == bool(s_ref) and abs(l2[i].item() - float(b_ref)) <= 1e-6
        same = ((adv[i:i + 1] - adv_ref).abs() <= 1e-6).float().mean().item()
        print(f"FGSM image {i}: success {bool(succ[i])} / ref {bool(s_ref)}, bound {l2[i].item()} / {b_ref}, identical pixels {100 * same:.2f}%")
        assert same >= 0.99
    assert bool(succ[0]) and l2[0].item() == 0.0 and torch.equal(adv[0], x[0])


def test_batched_apgd_runs_on_the_defense():
    from gen_adversarial_b200.nvae_spec import NvaeSpec, tiny_config
    from gen_adversarial_b200.defenses.ours.models import NVAEDefenseModel, CelebaIdentityClassifier
    from gen_adversarial_b200.defenses.wrappers import EoTWrapper
    cfg, res = tiny_config(initial_channels=16, groups=2, scales=2, latent=4), (3, 32, 32)
    spec = NvaeSpec(cfg, res)
    clf = CelebaIdentityClassifier({"state_dict": synth.make_vgg11_state_dict(10, seed=3, device=DEV)}, DEV, mode="bf16", n_classes=10, image_size=32)
    dm = NVAEDefenseModel(clf, synth.make_nvae_checkpoint(cfg, res, seed=3), [0.3] * spec.n_latents, 1.0, 0.5, False, DEV, mode="bf16").eval()
    x = synth.synthetic_batch(4, res, 10, seed=5)[0].to(DEV)
    with torch.no_grad():
        y = dm(x).argmax(1)
    for net in (dm, EoTWrapper(dm, 4)):                           # fused primitive, and torch autograd through the batched EoT wrapper
        succ, l2, adv = APGDL2(8, 0.75, 1.0)(x, y, net)
        assert succ.shape == (4,) and succ.dtype == torch.bool
        assert l2.max().item() <= 1.0 + 1e-4 and adv.min().item() >= 0 and adv.max().item() <= 1
        assert (adv - x).abs().max().item() > 1e-3
    lg = torch.randn(7, 6, device=DEV)
    assert dlr_loss(lg, lg.argmax(1)).shape == (7,)
