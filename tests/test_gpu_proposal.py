"""GPU parity of the proposal-sampling stage (SURVEY.md section 8a row A13) against the oracle."""
import pytest
import torch

from fruitnerf_b200 import _lib as L
from fruitnerf_b200 import ops
from fruitnerf_b200 import synthetic as syn
from fruitnerf_b200.compat import RayBundle, SceneBox, Semantics
from fruitnerf_b200.density_field import HashMLPDensityField
from fruitnerf_b200.fruit_field import SceneContraction
from fruitnerf_b200.fruit_nerf import FruitModel, FruitNerfModelConfig
from oracle import fruit_ref as fr
from oracle import ns_torch as ns

from .util import assert_rel

pytestmark = pytest.mark.gpu
AABB = torch.tensor([[-1.0, -1, -1], [1, 1, 1]])


def _net(sd, spec, dev):
    net = HashMLPDensityField(AABB, hidden_dim=spec.hidden_dim, log2_hashmap_size=spec.log2_hashmap_size, num_levels=spec.num_levels,
                              max_res=spec.max_res, spatial_distortion=SceneContraction())
    missing, unexpected = net.load_state_dict(sd, strict=False)
    assert not unexpected and all(k.startswith("mlp_base.0") or k in ("max_res", "num_levels", "log2_hashmap_size") for k in missing)
    return net.to(dev)


def _rays(R, salt=0):
    o, d, _, _, _ = syn.ray_batch(R, 4, salt=salt)
    return o, d, torch.full((R, 1), 0.05), torch.full((R, 1), 30.0)


@pytest.mark.parametrize("levels,max_res,S", [(5, 128, 256), (7, 2048, 96), (5, 256, 37)])
def test_proposal_weights_forward_backward(native_lib, cuda_device, levels, max_res, S):
    spec = fr.DensitySpec(num_levels=levels, max_res=max_res, log2_hashmap_size=15)
    sd = syn.density_state(num_levels=levels, log2_hashmap_size=15)
    net = _net(sd, spec, cuda_device)
    R = 48
    o, d, nears, fars = _rays(R, salt=2)
    bins = ns.spaced_bins(R, S, (syn.hash_uniform(R, 77).view(R, 1) + 1) * 0.5)
    e = ns.spacing_to_euclidean(bins, nears, fars)
    starts, ends = e[:, :-1].contiguous(), e[:, 1:].contiguous()
    coef = (syn.hash_uniform(R * S, 91).view(R, S) + 1.5)

    # gradient reference in float64: with 256 samples out to t = 30 the sums are ill-conditioned enough that the
    # oracle's own fp32 gradients deviate from the float64 ones by up to 1e-3 of the tensor scale
    spec64 = fr.DensitySpec(num_levels=levels, max_res=max_res, log2_hashmap_size=15)
    spec64.scalings = lambda: ns.hash_scalings(levels, 16, max_res).double()
    sd_ref = {k: v.double().clone().requires_grad_(k != "aabb") for k, v in sd.items()}
    w_ref = fr.proposal_weights(sd_ref, spec64, o.double(), d.double(), starts.double(), ends.double(), AABB.double())
    (w_ref * coef.double()).sum().backward()

    w = net.weights(o.cuda(), d.cuda(), starts.cuda(), ends.cuda())
    assert_rel(w, w_ref, what="proposal weights")
    (w * coef.cuda()).sum().backward()
    named = dict(net.named_parameters())
    for key in ("encoding.hash_table", "mlp_base.1.layers.0.weight", "mlp_base.1.layers.0.bias", "mlp_base.1.layers.1.weight",
                "mlp_base.1.layers.1.bias"):
        assert_rel(named[key].grad, sd_ref[key].grad, rel=3e-3, floor=0.5, what=f"grad {key}")


@pytest.mark.parametrize("mode", ["eval", "single_jitter", "per_bin"])
@pytest.mark.parametrize("S,n,anneal", [(256, 96, 1.0), (96, 48, 0.37), (64, 200, 1.0)])
def test_pdf_sample_matches_oracle(native_lib, cuda_device, mode, S, n, anneal):
    R = 64
    w = (syn.hash_uniform(R * S, 5).view(R, S) + 1.0).pow(6) * 0.01
    w[3] = 0.0  # zero-weight ray: the reference's eps padding path
    w[4, : S // 2] = 0.0
    existing = ns.spaced_bins(R, S, (syn.hash_uniform(R, 6).view(R, 1) + 1) * 0.5).contiguous()
    nears, fars = torch.full((R, 1), 0.05), torch.full((R, 1), 1000.0)
    u = None
    if mode == "single_jitter":
        u = (syn.hash_uniform(R, 8).view(R, 1) + 1) * 0.5
    elif mode == "per_bin":
        u = (syn.hash_uniform(R * (n + 1), 9).view(R, n + 1) + 1) * 0.5
    ref_bins = ns.pdf_sample(torch.pow(w, anneal), existing, n, u)
    bins, starts, ends = ops.pdf_sample(w.cuda(), existing.cuda(), n, None if u is None else u.cuda(), anneal, nears.cuda(), fars.cuda())
    # positions are continuous in u, so searchsorted ties only move a bin by rounding noise
    assert torch.allclose(bins.cpu(), ref_bins, atol=2e-6, rtol=1e-5), float((bins.cpu() - ref_bins).abs().max())
    e_ref = ns.spacing_to_euclidean(ref_bins, nears, fars)
    assert torch.allclose(starts.cpu(), e_ref[:, :-1], rtol=2e-4, atol=1e-6) and torch.allclose(ends.cpu(), e_ref[:, 1:], rtol=2e-4, atol=1e-6)
    assert bool((bins[:, 1:] >= bins[:, :-1]).all()), "bins must be sorted"


def test_interlevel_loss_value_and_gradient(native_lib, cuda_device):
    R = 96
    c = torch.sort(torch.cat([torch.zeros(R, 1), (syn.hash_uniform(R * 47, 1).view(R, 47) + 1) * 0.5, torch.ones(R, 1)], 1), 1).values
    w = torch.softmax(syn.hash_uniform(R * 48, 2).view(R, 48) * 3, -1) * 0.9
    levels = []
    for k, Sp in enumerate((256, 96)):
        cp = torch.sort(torch.cat([torch.zeros(R, 1), (syn.hash_uniform(R * (Sp - 1), 10 + k).view(R, Sp - 1) + 1) * 0.5, torch.ones(R, 1)], 1), 1).values
        wp = (torch.softmax(syn.hash_uniform(R * Sp, 20 + k).view(R, Sp) * 2, -1) * 0.8).requires_grad_(True)
        levels.append((cp, wp))
    ref = ns.interlevel_loss([wp for _, wp in levels] + [w], [cp for cp, _ in levels] + [c])
    ref.backward()
    gw = [wp.detach().cuda().requires_grad_(True) for _, wp in levels]
    out = ops.interlevel_loss(gw + [w.cuda()], [cp.cuda() for cp, _ in levels] + [c.cuda()], 1.0)
    out.backward()
    assert_rel(out.detach(), ref.detach(), what="interlevel loss")
    for g, (_, wp) in zip(gw, levels):
        assert_rel(g.grad, wp.grad, rel=2e-3, floor=0.05, what="d interlevel / d wp")


def test_model_eval_matches_oracle_pipeline(native_lib, cuda_device):
    """FruitModel.get_outputs in eval mode (deterministic sampler) vs the oracle's sampler + field + renderers."""
    cfg = FruitNerfModelConfig(log2_hashmap_size=15, use_average_appearance_embedding=False,
                               proposal_net_args_list=[
                                   {"hidden_dim": 16, "log2_hashmap_size": 14, "num_levels": 5, "max_res": 128, "use_linear": False},
                                   {"hidden_dim": 16, "log2_hashmap_size": 14, "num_levels": 5, "max_res": 256, "use_linear": False}])
    sem = Semantics(filenames=[], classes=["fruit"], colors=torch.tensor([[0.0, 0, 0], [1.0, 0, 0]]))
    model = FruitModel(cfg, metadata={"semantics": sem}, scene_box=SceneBox(AABB), num_train_data=7, test_mode="val")
    fsd = syn.field_state(log2_hashmap_size=15, num_images=7, table_scale=0.5, weight_gain=1.5)
    model.field.load_state_dict(fsd, strict=False)
    psd, pspecs = [], []
    for i, net in enumerate(model.proposal_networks):
        sd = syn.density_state(num_levels=5, log2_hashmap_size=14, salt=6000 + 100 * i, table_scale=1.0, weight_gain=2.0)
        net.load_state_dict(sd, strict=False)
        psd.append(sd)
        pspecs.append(fr.DensitySpec(num_levels=5, max_res=(128, 256)[i], log2_hashmap_size=14))
    model = model.to(cuda_device).eval()
    R = 64
    o, d, nears, fars = _rays(R, salt=4)
    rb = RayBundle(origins=o.cuda(), directions=d.cuda(), camera_indices=torch.zeros(R, 1, dtype=torch.long, device=cuda_device),
                   nears=nears.cuda(), fars=fars.cuda())
    with torch.no_grad():
        out = model(rb)
    assert len(out["weights_list"]) == 3 and len(out["ray_samples_list"]) == 3
    assert out["weights_list"][0].shape == (R, 256, 1) and out["weights_list"][1].shape == (R, 96, 1) and out["weights_list"][2].shape == (R, 48, 1)
    assert {"rgb", "accumulation", "depth", "semantics", "semantics_colormap", "prop_depth_0", "prop_depth_1"} <= set(out)
    starts, ends, bins, wl, sl = fr.proposal_sampler(psd, pspecs, o, d, nears, fars, (256, 96), 48, AABB)
    for k in range(2):
        assert_rel(out["weights_list"][k][..., 0], wl[k], what=f"proposal weights level {k}")
    assert torch.allclose(out["ray_samples_list"][2].frustums.starts[..., 0].cpu(), starts, rtol=5e-4, atol=1e-5)
    spec = fr.FieldSpec(log2_hashmap_size=15)
    f = fr.field_forward(fsd, spec, o[:, None, :], d[:, None, :], starts[..., None], ends[..., None], None, True, "zeros")
    ref = fr.render(f, starts[..., None], ends[..., None], training=False)
    # the final bins differ by rounding noise (1e-4 rel on far bins), which the hash grid amplifies mildly: compare at 5e-3
    assert_rel(out["rgb"], ref["rgb"], rel=5e-3, what="rgb")
    assert_rel(out["semantics"], ref["semantics"], rel=5e-3, what="semantics")


def test_model_train_step_produces_all_gradients(native_lib, cuda_device):
    # the random initialisation decides whether proposal level 0 gets any interlevel gradient: for some draws its outer bound
    # already covers every fine weight (loss term and gradient exactly 0, in the oracle too), so the test must not inherit
    # whatever RNG state the tests before it left behind
    torch.manual_seed(0)
    cfg = FruitNerfModelConfig(log2_hashmap_size=15, proposal_net_args_list=[
        {"hidden_dim": 16, "log2_hashmap_size": 14, "num_levels": 5, "max_res": 128, "use_linear": False},
        {"hidden_dim": 16, "log2_hashmap_size": 14, "num_levels": 5, "max_res": 256, "use_linear": False}])
    sem = Semantics(filenames=[], classes=["fruit"], colors=torch.tensor([[0.0, 0, 0], [1.0, 0, 0]]))
    model = FruitModel(cfg, metadata={"semantics": sem}, scene_box=SceneBox(AABB), num_train_data=7, test_mode="val").to(cuda_device).train()
    with torch.no_grad():
        model.field.mlp_base_grid.hash_table.mul_(300.0)
        for net in model.proposal_networks:
            net.encoding.hash_table.mul_(300.0)
    R = 128
    o, d, nears, fars = _rays(R, salt=6)
    img, mask = syn.targets(R)
    rb = RayBundle(origins=o.cuda(), directions=d.cuda(), camera_indices=torch.randint(0, 7, (R, 1), device=cuda_device),
                   nears=nears.cuda(), fars=fars.cuda())
    for cb in model.get_training_callbacks():
        if cb["where_to_run"] == "BEFORE_TRAIN_ITERATION":
            cb["func"](0)
    out = model(rb)
    batch = {"image": img.cuda(), "fruit_mask": mask.cuda()}
    losses = model.get_loss_dict(out, batch)
    assert set(losses) == {"rgb_loss", "semantics_loss", "interlevel_loss"}
    sum(losses.values()).backward()
    metrics = model.get_metrics_dict(out, batch)
    assert torch.isfinite(metrics["psnr"]) and torch.isfinite(metrics["distortion"])
    for name, p in model.named_parameters():
        if name == "device_indicator_param" or name.startswith("field.mlp_base.") or ".mlp_base.0." in name:
            continue
        assert p.grad is not None and torch.isfinite(p.grad).all(), name
    assert float(model.proposal_networks[0].encoding.hash_table.grad.abs().sum()) > 0
    assert float(model.field.mlp_base_grid.hash_table.grad.abs().sum()) > 0
