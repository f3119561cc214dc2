#!/usr/bin/env python
"""More fixtures from the UNMODIFIED reference (build container only, same shims as make_golden.py):

  gen_<case>.pt        the reference's own ``P2PModel.p2p_generate`` (models/p2p_model.py:80-183) in eval mode
                       (BatchNorm on its running statistics), for model_mode in {full, posterior, prior} x skip_frame in
                       {False, True}: inputs, NumPy skip draws, the eps stream, BN buffers, every generated frame as a
                       digest and the last frame in full.
  ckpt_ref_small.pth   a checkpoint written by the reference's own ``P2PModel.save`` (models/p2p_model.py:289-308) after
                       one training step of a SMALL configuration (h36m_mlp backbone, g_dim 32, rnn_size 32: a few
                       hundred KB; the checkpoint format does not depend on the backbone)
  ckpt_ref_small_next.pt   the batch / eps / skip draws and the four losses of the reference's NEXT step from that
                       checkpoint (resume check), plus digests of the checkpointed tensors.
  ckpt_ref_resume.pt   the reverse direction: a checkpoint written by the drop-in ``P2PModel.save`` (ckpt_ref_small.pth
                       loaded, saved as epoch 9) loaded by the reference's own ``P2PModel.load`` under stock
                       ``torch.optim.Adam``, then one Adam step with all gradients set to one.  Stores the reference's
                       module layout (state_dict keys / shapes, parameter order), the epoch ``load`` returned, and the
                       Adam step counts and digests of the parameters after that step.
  init_sha256.json     for every case of make_golden.py, the SHA-256 of each floating-point tensor of the reference's
                       freshly initialised modules (float32 bytes): pins the initial weights bit for bit, whatever order
                       a sum over them would be taken in.

    python tests/golden/make_golden_extra.py [gen] [ckpt] [resume] [init]     (default: all)
"""
import hashlib
import json
import os
import subprocess
import sys
import tempfile

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
from make_golden import CASES, LegacyAdam, ROOT, import_reference, make_opt  # noqa: E402

sys.path.insert(0, ROOT)
from oracle.p2p_oracle import tensor_digest  # noqa: E402

GEN_CASES = {
    # n_past = 1 (the training default): ground truth is only the first frame
    "d64": dict(width=64, channels=1, T_in=5, len_output=7, B=2, opt=dict(skip_prob=0.5)),
    # n_past = 2 + last_frame_skip: the `i < n_past` branch (posterior / prior advance on ground truth) and fresh skips
    "d64_np2": dict(width=64, channels=1, T_in=4, len_output=6, B=2, opt=dict(skip_prob=0.5, n_past=2, last_frame_skip=True)),
}


def warm_bn(model, spec, gen):
    """Move the BatchNorm running statistics off their initial (0, 1) without touching any weight: a few train-mode
    forward calls of the reference's own encoder / decoder under no_grad."""
    model.train()
    with torch.no_grad():
        for _ in range(3):
            xb = torch.rand(4, spec["channels"], spec["width"], spec["width"], generator=gen)
            h, skips = model.encoder(xb)
            model.decoder([torch.tanh(torch.randn(4, 128, generator=gen)), skips])
    model.eval()


def run_gen_case(name, spec, p2p_model, backbones):
    torch.manual_seed(1)
    opt = make_opt(backbones[spec["width"]], batch_size=spec["B"], **spec["opt"])
    model = p2p_model.P2PModel(opt.batch_size, spec["channels"], 128, 10, 256, 1, 1, 2, opt=opt)
    gen = torch.Generator().manual_seed(4321)
    warm_bn(model, spec, gen)
    x = torch.rand(spec["T_in"], spec["B"], spec["channels"], spec["width"], spec["width"], generator=gen)
    mods = dict(encoder=model.encoder, decoder=model.decoder)
    fix = dict(case=name, init_seed=1, cfg=dict(g_dim=128, z_dim=10, rnn_size=256, channels=spec["channels"], image_width=spec["width"],
                                                 predictor_rnn_layers=2, posterior_rnn_layers=1, prior_rnn_layers=1),
               opt={k: getattr(opt, k) for k in ("beta", "weight_cpc", "weight_align", "skip_prob", "n_past", "last_frame_skip", "lr",
                                                 "beta1", "batch_size")},
               x=x, len_output=spec["len_output"], eval_cp_ix=spec["len_output"] - 1,
               bn_buffers={m: {k: v.detach().clone() for k, v in mods[m].state_dict().items() if "running_" in k or "num_batches" in k}
                           for m in mods},
               runs=[])
    n_calls = []
    hook = model.posterior.register_forward_hook(lambda *a: n_calls.append(1))
    for mode in ("full", "posterior", "prior"):
        for skip_frame in (False, True):
            seed = 100 + len(fix["runs"])
            np.random.seed(seed)
            probs = np.random.uniform(0, 1, spec["len_output"] - 1)
            np.random.seed(seed)
            torch.manual_seed(seed)
            n_calls.clear()
            with torch.no_grad():
                seq = model.p2p_generate(x, spec["len_output"], spec["len_output"] - 1, model_mode=mode, skip_frame=skip_frame)
            n_exec = len(n_calls)
            torch.manual_seed(seed)
            eps = torch.empty(n_exec, 2, spec["B"], 10)
            for s in range(n_exec):
                eps[s, 0].normal_()
                eps[s, 1].normal_()
            zeros = [bool((f == 0).all()) for f in seq]
            fix["runs"].append(dict(model_mode=mode, skip_frame=skip_frame, np_seed=seed, probs=torch.from_numpy(probs), eps=eps,
                                    n_exec=n_exec, zero_frames=zeros, digests=[tensor_digest(f) for f in seq],
                                    last=seq[-1].detach().clone(), mid=seq[len(seq) // 2].detach().clone()))
            print(f"[gen_{name}] mode={mode} skip_frame={skip_frame}: executed {n_exec}, zero frames {zeros}")
    hook.remove()
    path = os.path.join(HERE, f"gen_{name}.pt")
    torch.save(fix, path)
    print("wrote", path, os.path.getsize(path) // 1024, "KiB")


def run_ckpt_case(p2p_model, backbones):
    torch.manual_seed(1)
    g_dim, z_dim, rnn, B, T = 32, 4, 32, 4, 5
    opt = make_opt(backbones["mlp"], dataset="h36m", batch_size=B)
    model = p2p_model.P2PModel(B, 1, g_dim, z_dim, rnn, 1, 1, 2, opt=opt)
    model.opt.optimizer = LegacyAdam
    model.init_optimizer()
    model.train()
    gen = torch.Generator().manual_seed(99)

    def step(seed):
        x = 3 * torch.randn(T, B, 17, 3, generator=gen)
        np.random.seed(seed)
        probs = np.random.uniform(0, 1, T - 1)
        np.random.seed(seed)
        torch.manual_seed(seed)
        model.zero_grad()
        losses = model((None, x, None), 0, T - 1)
        torch.manual_seed(seed)
        eps = torch.empty(T - 1, 2, B, z_dim)
        for s in range(T - 1):
            eps[s, 0].normal_()
            eps[s, 1].normal_()
        return x, probs, eps, [float(v) for v in losses]

    step(7)
    path = os.path.join(HERE, "ckpt_ref_small.pth")
    # a real reference checkpoint pickles opt.optimizer = torch.optim.Adam (models/p2p_model.py:41); the Mode-A shim class
    # lives in this script and must not leak into the file
    model.opt.optimizer = torch.optim.Adam
    model.save(path, 3)   # the reference's own save(): epoch 3
    model.opt.optimizer = LegacyAdam
    mods = ("frame_predictor", "posterior", "prior", "encoder", "decoder")
    digests = {m: {k: tensor_digest(v) for k, v in getattr(model, m).state_dict().items() if v.is_floating_point()} for m in mods}
    x, probs, eps, losses = step(8)
    side = dict(cfg=dict(g_dim=g_dim, z_dim=z_dim, rnn_size=rnn, backbone="mlp", predictor_rnn_layers=2, posterior_rnn_layers=1,
                         prior_rnn_layers=1),
                B=B, T=T, epoch=3, digests=digests, next=dict(x=x, probs=torch.from_numpy(probs), eps=eps, losses=losses),
                post_digests={m: {k: tensor_digest(v) for k, v in getattr(model, m).state_dict().items() if v.is_floating_point()}
                              for m in mods})
    torch.save(side, os.path.join(HERE, "ckpt_ref_small_next.pt"))
    print("wrote", path, os.path.getsize(path) // 1024, "KiB; next-step losses", losses)


def run_resume_case(p2p_model, backbones):
    with tempfile.TemporaryDirectory() as tmp:
        dropin_pth = os.path.join(tmp, "dropin.pth")
        # the drop-in and the reference both own the package names `models` / `misc`: write the drop-in checkpoint in a
        # process of its own
        subprocess.check_call([sys.executable, "-c", "import sys; sys.path.insert(0, sys.argv[1]); "
                               "from tests.test_generate_ckpt_golden import small_model, GOLD; import os; m, _ = small_model(); "
                               "m.load(os.path.join(GOLD, 'ckpt_ref_small.pth')); m.save(sys.argv[2], 9)", ROOT, dropin_pth])
        states = torch.load(dropin_pth, weights_only=False)
    side = torch.load(os.path.join(HERE, "ckpt_ref_small_next.pt"), weights_only=False)
    cfg, B = side["cfg"], side["B"]
    torch.manual_seed(11)
    opt = make_opt(backbones["mlp"], dataset="h36m", batch_size=B)
    model = p2p_model.P2PModel(B, 1, cfg["g_dim"], cfg["z_dim"], cfg["rnn_size"], 1, 1, 2, opt=opt)   # stock torch.optim.Adam
    mods = ("frame_predictor", "posterior", "prior", "encoder", "decoder")
    layout = {m: dict(state=[(k, tuple(v.shape)) for k, v in getattr(model, m).state_dict().items()],
                      params=[k for k, _ in getattr(model, m).named_parameters()]) for m in mods}
    # torch >= 2.6 defaults torch.load to weights_only=True, which the reference's load(pth) does not survive for a
    # checkpoint carrying the pickled opt namespace: hand it the states instead
    epoch = model.load(states=states)
    adam = {}
    for m in mods:
        o = getattr(model, m + "_optimizer")
        assert type(o) is torch.optim.Adam
        adam[m] = dict(lr=o.param_groups[0]["lr"], betas=tuple(o.param_groups[0]["betas"]))
        for p in getattr(model, m).parameters():
            p.grad = torch.ones_like(p)
        o.step()
    fix = dict(cfg=cfg, B=B, saved_epoch=9, start_epoch=epoch, layout=layout, adam=adam,
               steps={m: [int(v["step"]) for v in getattr(model, m + "_optimizer").state_dict()["state"].values()] for m in mods},
               post={m: {k: tensor_digest(v) for k, v in getattr(model, m).named_parameters()} for m in mods})
    path = os.path.join(HERE, "ckpt_ref_resume.pt")
    torch.save(fix, path)
    print("wrote", path, os.path.getsize(path) // 1024, "KiB; start epoch", epoch)


def sha256_f32(t):
    return hashlib.sha256(t.detach().to(torch.float32).contiguous().numpy().tobytes()).hexdigest()


def run_init_case(p2p_model, backbones):
    out = {}
    for name, spec in CASES.items():
        torch.manual_seed(1)   # the construction of make_golden.run_case
        opt = make_opt(backbones[spec["width"]], **spec["opt"])
        if opt.batch_size is None:
            opt.batch_size = spec["B"]
        model = p2p_model.P2PModel(opt.batch_size, spec["channels"], 128, 10, 256, 1, 1, 2, opt=opt)
        out[name] = {m: {k: sha256_f32(v) for k, v in getattr(model, m).state_dict().items() if v.is_floating_point()}
                     for m in ("frame_predictor", "posterior", "prior", "encoder", "decoder")}
    path = os.path.join(HERE, "init_sha256.json")
    with open(path, "w") as f:
        json.dump(out, f, indent=0, sort_keys=True)
    print("wrote", path, os.path.getsize(path) // 1024, "KiB")


def main():
    parts = sys.argv[1:] or ["gen", "ckpt", "resume", "init"]
    torch.set_num_threads(8)
    p2p_model, backbones = import_reference()
    if "gen" in parts:
        for name, spec in GEN_CASES.items():
            run_gen_case(name, spec, p2p_model, backbones)
    if "ckpt" in parts:
        run_ckpt_case(p2p_model, backbones)
    if "resume" in parts:
        run_resume_case(p2p_model, backbones)
    if "init" in parts:
        run_init_case(p2p_model, backbones)


if __name__ == "__main__":
    main()
