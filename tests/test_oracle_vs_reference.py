"""CPU: the oracle port against the unmodified reference (gaopinghai/BDE2VID).

When the reference's tree is reachable (``BDE2VID_REFERENCE``, see oracle/ref_shim.py) every test runs the reference
itself and asks for bit-equal results.  Otherwise the same inputs are checked against tests/golden/reference_live.npz:
the outputs of the oracle port on exactly these inputs, recorded from the oracle as commit 5f45621 left it (the commit
that wrote these tests to hold it bit-equal to the live reference; the oracle has not changed since), and the key /
shape sets of the state dicts the reference's strict load accepted.  On other hosts fp32 sums may reassociate, so the stored frames are compared
with the tolerance of test_oracle_golden.py; voxel grids and the percentile norm stay bit-exact."""
import numpy as np
import pytest
import torch

from bde2vid_b200 import synth
from conftest import load_golden
from oracle import oracle_torch as O
from oracle import ref_shim

LIVE = ref_shim.reference_available()
VARIANTS = [dict(recurrent_block_type="convgru", skip_type="concat", depths=[1, 0, 0], num_res_blocks=1),
            dict(norm="BN", nwindow_size=(2, 3), depths=[1, 0, 1], useRC=False)]


def _keys(sd):
    return sorted("%s:%s" % (k, "x".join(map(str, v.shape))) for k, v in sd.items())


def _check_forward(cfg, sd, vox, name):
    """The oracle's frames on ``vox`` against the reference's, and ``sd`` strictly loadable into the reference model."""
    with torch.no_grad():
        mine = torch.cat(O.bde2vid_forward(sd, cfg, vox), 0)
    if LIVE:
        R = ref_shim.reference_modules()
        model = R.BDE2VID(generator=dict(cfg)).eval()
        model.load_state_dict(sd, strict=True)
        with ref_shim.cpu_mode(), torch.no_grad():
            ref = torch.cat(model([{"events": v} for v in vox]), 0)
        assert float((ref - mine).abs().max()) == 0.0
    else:
        g = load_golden("reference_live")
        assert _keys(sd) == list(g[name + "_keys"])
        assert np.abs(mine.numpy() - g[name + "_frames"]).max() <= 2e-6


def test_voxel_vs_reference():
    ev = synth.gen_events(11, 2, 90, 120, 4000)
    for w in range(2):
        xs, ys, ts, ps = synth.to_loader_format(ev, w)
        if LIVE:
            R = ref_shim.reference_modules()
            ref = R.events_to_voxel_torch(*(torch.from_numpy(a) for a in (xs, ys, ts, ps)), 5, sensor_size=(90, 120)).numpy()
        else:
            ref = load_golden("reference_live")["voxel_w%d" % w]
        assert np.array_equal(ref, O.voxel_grid(xs, ys, ts, ps, 5, (90, 120)))


def test_bde2vid_vs_reference_and_strict_load():
    cfg = O.full_cfg()
    sd = synth.init_state_dict(cfg, 5, stress=True)     # our synthetic checkpoints carry the reference's exact key set
    g = torch.Generator().manual_seed(3)
    vox = [torch.randn(1, 5, 56, 64, generator=g) for _ in range(3)]
    _check_forward(cfg, sd, vox, "bde2vid")


@pytest.mark.parametrize("over", VARIANTS)
def test_variants_vs_reference_live(over):
    """Variant cfgs not in the other goldens: strict load of our container's keys into the reference model, oracle
    bit-equal to the reference forward."""
    from bde2vid_b200.model import BDE2VID
    cfg = O.full_cfg(over)
    ours = BDE2VID(generator=dict(cfg))
    sd = synth.random_state_dict_like(ours.state_dict(), 77)
    g = torch.Generator().manual_seed(4)
    vox = [torch.randn(1, 5, 56, 64, generator=g) for _ in range(3)]
    _check_forward(cfg, sd, vox, "variant%d" % VARIANTS.index(over))


def test_loader_transforms_vs_reference_live():
    ev = synth.gen_events(61, 1, 40, 56, 2500)
    v = torch.from_numpy(O.voxel_grid(*synth.to_loader_format(ev, 0), 5, (40, 56)))
    legacy, robust = O.legacy_norm(v.clone()), O.robust_norm(v.clone(), 2, 98)
    if LIVE:
        ref_shim.install()
        from utils_func.data_augmentation import LegacyNorm
        from utils_func.utils import RobustNorm
        assert torch.equal(LegacyNorm()(v.clone()), legacy)
        assert torch.equal(RobustNorm(2, 98)(v.clone()), robust)
    else:
        g = load_golden("reference_live")
        assert np.abs(legacy.numpy() - g["legacy_norm"]).max() <= 1e-5     # mean / std are fp32 sums
        assert np.array_equal(robust.numpy(), g["robust_norm"])
