"""CPU: host-side logic of the drop-in (no kernels): pad/crop geometry, registry + config loading path,
state_dict compatibility with the reference key set, window maps, weight packing, sharding."""
import pytest
import torch

from bde2vid_b200 import synth
from bde2vid_b200.croper import Croper
from bde2vid_b200.dist import finalize_means, shard_units
from bde2vid_b200.engine import _pack_conv, window_token_map
from bde2vid_b200.model import BDE2VID, MODELS
from bde2vid_b200.registry import Config
from oracle import oracle_torch as O


def test_croper_matches_reference_fixture(manifest):
    for key, rec in manifest["croper"].items():
        wh, e = key.split("_e")
        w, h = [int(v) for v in wh.split("x")]
        c = Croper(int(e))
        c.update_params(w, h)
        assert [c.height_crop_size, c.width_crop_size] == [rec["Hp"], rec["Wp"]]
        assert [c.padding_left, c.padding_right, c.padding_top, c.padding_bottom] == rec["pad"]
        assert [c.iy0, c.iy1, c.ix0, c.ix1] == rec["crop"]
        x = torch.arange(h * w, dtype=torch.float32).reshape(1, 1, h, w)
        assert torch.equal(c.crop(c.pad(x)), x)


def test_checkpoint_loading_path_and_key_compat():
    """eval_models_seq.py:52-60,:86: Config.fromstring(meta.cfg).model -> MODELS.build -> load_state_dict(strict)."""
    cfg = Config.fromstring(synth.ASSUMED_CFG_STR, ".py").model
    assert cfg["type"] == "BDE2VID" and cfg.generator["num_bins"] == 5
    model = MODELS.build(cfg)
    assert isinstance(model, BDE2VID)
    sd = synth.init_state_dict(cfg["generator"], 0)
    assert len(sd) == 220 and sum(v.numel() for v in sd.values()) == 21086523      # SURVEY.md section 8
    assert list(model.state_dict().keys()) == list(sd.keys())
    model.load_state_dict(sd, strict=True)
    assert hasattr(model, "reset_states") and model.cpu_cache_length == 100
    model.reset_states()


def test_unsupported_configs_raise_not_fallback():
    """What the sm_100a path does not build raises at construction (never a CPU path); every architecture option of
    the reference constructor that IS built constructs."""
    base = dict(Config.fromstring(synth.ASSUMED_CFG_STR, ".py").model["generator"])
    for bad in (dict(norm="GN"), dict(skip_type="no_skip"), dict(num_output_channels=3), dict(act_net="ELU"),
                dict(activation=dict(type="LReLU"))):
        with pytest.raises(NotImplementedError):
            BDE2VID(generator=dict(base, **bad))
    for ok in (dict(norm="BN"), dict(norm="IN"), dict(recurrent_block_type="convgru"), dict(skip_type="concat"),
               dict(nwindow_size=(3, 3)), dict(depths=[4, 0, 0]), dict(useRC=False), dict(activation=dict(type="Identity"))):
        BDE2VID(generator=dict(base, **ok))
    m = BDE2VID(generator=base)
    with pytest.raises(NotImplementedError):
        m([], mode="loss")


def test_plan_cache_is_bounded():
    """Engine.plans is an LRU bounded in bytes (the driver with subseq_L=None calls the model with a new T per file)."""
    from collections import OrderedDict
    from bde2vid_b200.engine import Engine

    class P:
        def __init__(self, n):
            self.nbytes, self.released = n, False

        def release(self):
            self.released = True

    eng = Engine.__new__(Engine)
    eng.plans, eng.plan_cache_bytes = OrderedDict(), 250
    made = []
    import bde2vid_b200.engine as E
    orig = E._Plan
    E._Plan = lambda e, T, B, Hp, Wp: made.append(P(100)) or made[-1]
    try:
        a = eng.plan(1, 1, 8, 8)
        b = eng.plan(2, 1, 8, 8)
        assert eng.plan(1, 1, 8, 8) is a                     # hit: moves to the MRU end
        c = eng.plan(3, 1, 8, 8)                             # 300 bytes > 250: evicts the LRU entry (b)
        assert b.released and not a.released and not c.released
        assert list(eng.plans.keys()) == [(1, 1, 8, 8, 0), (3, 1, 8, 8, 0)]
        eng.plan_cache_bytes = 50
        d = eng.plan(4, 1, 8, 8)                             # a single plan larger than the budget still lives
        assert list(eng.plans.values()) == [d] and a.released and c.released
    finally:
        E._Plan = orig


@pytest.mark.parametrize("H,W", [(12, 20), (9, 13), (7, 30), (33, 44), (132, 176)])
def test_window_token_map_matches_oracle(H, W):
    for dil in (False, True):
        mine, _ = window_token_map(2, H, W, (7, 7), dil, "cpu")
        idx, ok, _ = O.window_token_map(H, W, dil)
        n = idx.shape[0]
        assert torch.equal(mine[:n].long(), idx)
        assert torch.equal(mine[n:].long(), torch.where(idx >= 0, idx + H * W, idx))
        # every real pixel is covered by at most one token (F.fold never sums on this path)
        flat = idx[idx >= 0]
        assert flat.numel() == flat.unique().numel()


def test_pack_conv_orders():
    w = torch.arange(2 * 128 * 3 * 3, dtype=torch.float32).reshape(2, 128, 3, 3)
    tap, ld = _pack_conv(w, torch.float32)
    cm, ld2 = _pack_conv(w, torch.float32, chunk_major=True)
    assert ld == ld2 == 1152
    for (co, ci, ky, kx) in [(0, 0, 0, 0), (1, 70, 2, 1), (0, 127, 1, 2)]:
        t = ky * 3 + kx
        assert tap[co, t * 128 + ci] == w[co, ci, ky, kx]
        assert cm[co, (ci // 64) * 9 * 64 + t * 64 + ci % 64] == w[co, ci, ky, kx]
    head, ldh = _pack_conv(torch.ones(32, 5, 5, 5), torch.float32, cin_pad=8)
    assert ldh == 256 and head[:, :200].reshape(32, 25, 8)[:, :, 5:].abs().sum() == 0


def test_shard_units_balanced_and_complete():
    costs = [100, 90, 80, 10, 10, 10, 5, 5]
    for world in (1, 2, 4, 8):
        parts = shard_units(costs, world)
        assert sorted(i for p in parts for i in p) == list(range(len(costs)))
        loads = [sum(costs[i] for i in p) for p in parts]
        assert max(loads) - min(loads) <= max(costs)
    assert finalize_means({"mse": 4.0, "ssim": 2.0, "n": 4.0}) == {"mse": 1.0, "ssim": 0.5}


def test_synthetic_events_follow_loader_contract():
    ev = synth.gen_events(3, 2, 20, 30, 100)
    assert ev["xs"].dtype.name == "int16" and ev["ts"].dtype.name == "float64" and ev["ps"].dtype.name == "bool"
    xs, ys, ts, ps = synth.to_loader_format(ev, 1)
    assert xs.dtype.name == "float32" and ts[0] == 0.0 and set(ps.tolist()) <= {-1.0, 1.0}
    assert (ts[1:] >= ts[:-1]).all() and xs.max() < 30 and ys.max() < 20


def test_e2vid_state_dict_keys_match_reference(manifest):
    """Strict load of a reference-layout E2VIDRecurrent checkpoint (keys recorded from the reference's own
    state_dict by oracle/make_golden.py)."""
    from bde2vid_b200.e2vid import E2VIDRecurrent
    rec = manifest["e2vid_64x96_B2_T3"]
    m = E2VIDRecurrent({"num_bins": 5})
    sd = m.state_dict()
    assert list(sd.keys()) == rec["keys"]
    assert [list(v.shape) for v in sd.values()] == rec["shapes"]
    assert m.num_encoders == 4


def test_bench_contract_without_gpu():
    """bench.py / bench_configs.py import cleanly, every --config has its runner, the product arm refuses to run without a
    CUDA device (no CPU fallback), and the reference arm prints one JSON line with the contract's keys on a tiny sample."""
    import json
    import os
    import subprocess
    import sys
    import bench
    import bench_configs
    for cfg in ("e2vid16", "gen4", "shard64", "pair"):
        assert callable(getattr(bench_configs, "run_" + cfg))
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    if not torch.cuda.is_available():
        r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--steps", "1", "--warmup", "1"], capture_output=True,
                           text=True, cwd=root)
        assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--ref-windows", "2"], capture_output=True, text=True, cwd=root, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
    assert line["impl"] == "reference" and line["unit"] == "frames/s" and line["higher_is_better"] is True
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0 and line["value"] > 0
    assert getattr(bench, "VOXEL_BYTES_PER_WINDOW") == 16 * 31500 + 4 * 5 * 260 * 346


def test_bench_dump_outputs(tmp_path, monkeypatch):
    """--dump-outputs: every frame of every sequence, whole when it fits the byte budget, else at the same seeded pixels."""
    import numpy as np
    import bench
    seqs = [[torch.rand(1, 1, 6, 7) for _ in range(4)] for _ in range(3)]
    full = torch.stack([torch.cat(s, 0) for s in seqs]).flatten(2).numpy()
    bench.dump_outputs(str(tmp_path / "all"), seqs)
    got = np.load(tmp_path / "all" / "frames.npy")
    assert got.dtype == np.float32 and np.array_equal(got, full)
    assert np.array_equal(np.load(tmp_path / "all" / "frame_pixels.npy"), np.arange(42))
    monkeypatch.setattr(bench, "DUMP_BYTES", 10 * (4 * 3 * 4 + 8))
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), seqs)
    pix = np.load(tmp_path / "a" / "frame_pixels.npy")
    got = np.load(tmp_path / "a" / "frames.npy")
    assert pix.dtype == np.float64 and len(set(pix)) == 10 and np.array_equal(pix, np.load(tmp_path / "b" / "frame_pixels.npy"))
    assert got.shape == (3, 4, 10) and np.array_equal(got, full[:, :, pix.astype(int)])
