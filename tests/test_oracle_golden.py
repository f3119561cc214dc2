"""Pin the oracle (oracle/p2p_oracle.py) against fixtures produced by the unmodified reference
(tests/golden/make_golden.py).  CPU only."""
import glob
import hashlib
import json
import os

import numpy as np
import pytest
import torch

from oracle import p2p_oracle as O

GOLD = os.path.join(os.path.dirname(__file__), "golden")
CASES = sorted(os.path.basename(p)[5:-3] for p in glob.glob(os.path.join(GOLD, "step_*.pt")))


def load(case):
    return torch.load(os.path.join(GOLD, f"step_{case}.pt"), weights_only=False)


def check_digest(t, d, rtol, atol, what):
    f = t.detach().double().reshape(-1)
    assert f.numel() == d["numel"], what
    got = f[d["idx"]]
    scale = max(d["absmax"], 1e-30)
    err = (got - d["samples"]).abs().max().item()
    assert err <= atol + rtol * scale, f"{what}: sample err {err:.3e} (scale {scale:.3e})"
    assert abs(float(f.norm()) - d["l2"]) <= atol + rtol * max(d["l2"], 1e-30), f"{what}: l2"


@pytest.mark.parametrize("case", CASES)
def test_initial_weights_bit_exact(case):
    """Samples against the step fixture, every element against the reference's SHA-256 (tests/golden/init_sha256.json):
    a float64 sum over the tensor would depend on the host's thread count and vector width."""
    fix = load(case)
    sha = json.load(open(os.path.join(GOLD, "init_sha256.json")))[case]
    state = O.build_state(fix["cfg"], seed=fix["init_seed"])
    for m, digs in fix["init_digest"].items():
        assert sorted(digs) == sorted(sha[m]), m
        for k, d in digs.items():
            f = state[m][k].double().reshape(-1)
            assert torch.equal(f[d["idx"]], d["samples"]), f"{m}.{k}"
            assert hashlib.sha256(state[m][k].to(torch.float32).contiguous().numpy().tobytes()).hexdigest() == sha[m][k], f"{m}.{k}"


@pytest.mark.parametrize("case", CASES)
def test_skip_schedule_bit_exact(case):
    fix = load(case)
    for rec in fix["steps"]:
        probs = rec["probs"].numpy()
        np.random.seed(rec["np_seed"])
        assert np.array_equal(np.random.uniform(0, 1, len(probs)), probs)
        sched = O.skip_schedule(rec["x"].shape[0], probs, fix["opt"]["skip_prob"], fix["opt"]["n_past"])
        posts = [r for r in rec["tape"] if r["m"] == "posterior"]
        assert len(sched) == rec["n_exec"] == len(posts)
        for (i, tuc, dt), r in zip(sched, posts):
            # columns 2g and 2g+1 of the posterior input hold the fp32-rounded counters
            g = fix["cfg"]["g_dim"]
            col_tuc, col_dt = r["inp"][:, 2 * g], r["inp"][:, 2 * g + 1]
            assert torch.equal(col_tuc, torch.full_like(col_tuc, tuc))
            assert torch.equal(col_dt, torch.full_like(col_dt, dt))


@pytest.mark.parametrize("case", CASES)
def test_train_step_matches_reference(case):
    fix = load(case)
    torch.set_num_threads(min(8, os.cpu_count() or 1))
    state = O.build_state(fix["cfg"], seed=fix["init_seed"])
    adam = {m: O.new_adam_state(state[m]) for m in O.MODULES}
    width = fix["cfg"]["image_width"]
    for rec in fix["steps"]:
        tape = []
        out = O.train_step(state, adam, rec["x"], fix["opt"], width, rec["eps"], rec["probs"].numpy(), mode="A", tape=tape)
        np.testing.assert_allclose(out["losses"], rec["losses"], rtol=2e-5, atol=1e-7)
        posts = [r for r in rec["tape"] if r["m"] == "posterior"]
        preds = [r for r in rec["tape"] if r["m"] == "frame_predictor"]
        for s, t in enumerate(tape):
            assert torch.allclose(t["mu"], posts[s]["mu"], rtol=1e-4, atol=1e-6)
            assert torch.allclose(t["logvar"], posts[s]["logvar"], rtol=1e-4, atol=1e-6)
            assert torch.allclose(t["h_pred"], preds[s]["out"], rtol=1e-4, atol=1e-6)
        for m, digs in rec["grad_digest"].items():
            for k, d in digs.items():
                check_digest(out["grads"][m][k], d, rtol=2e-4, atol=1e-9, what=f"grad {m}.{k}")
        for m, digs in rec["post_digest"].items():
            for k, d in digs.items():
                check_digest(state[m][k], d, rtol=2e-5, atol=1e-8, what=f"post {m}.{k}")
        for m, bufs in rec["bn_buffers"].items():
            for k, v in bufs.items():
                if v.is_floating_point():
                    assert torch.allclose(state[m][k], v, rtol=1e-5, atol=1e-7), f"{m}.{k}"
                else:
                    assert torch.equal(state[m][k], v), f"{m}.{k}"


def test_mode_b_differs_only_in_prior():
    fix = load("d64_plain")
    rec = fix["steps"][0]
    width = fix["cfg"]["image_width"]
    res = {}
    for mode in ("A", "B"):
        state = O.build_state(fix["cfg"], seed=fix["init_seed"])
        adam = {m: O.new_adam_state(state[m]) for m in O.MODULES}
        res[mode] = O.train_step(state, adam, rec["x"], fix["opt"], width, rec["eps"], rec["probs"].numpy(), mode=mode)
    assert res["A"]["losses"] == res["B"]["losses"]
    for m in ("encoder", "decoder", "posterior", "frame_predictor"):
        for k, g in res["A"]["grads"][m].items():
            assert torch.equal(g, res["B"]["grads"][m][k])
    diff = max((res["A"]["grads"]["prior"][k] - res["B"]["grads"]["prior"][k]).abs().max().item() for k in res["A"]["grads"]["prior"])
    assert diff > 0
