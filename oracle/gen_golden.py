"""Generate tests/golden/*.npz|json by running the REAL reference (TEST INFRASTRUCTURE; needs a reference checkout).

Imports the reference's own modules from the checkout FDM_B200_REFERENCE_DIR names, with the harness shims of
SURVEY.md §8(c), gives them the deterministic weights of oracle/weights.py, and records (a) their state_dict layout,
(b) their outputs on seeded inputs. While doing so it checks the oracle restatement (oracle/reference_ops.py) against
the reference and refuses to write fixtures if they disagree. The tests need only the committed fixtures, not the
reference.

    FDM_B200_REFERENCE_DIR=<reference checkout> python oracle/gen_golden.py     # writes tests/golden/
"""
import json
import os
import sys
import types

import numpy as np
import torch

REF = os.environ.get("FDM_B200_REFERENCE_DIR", "")
if not os.path.isdir(REF):
    sys.exit("usage: FDM_B200_REFERENCE_DIR=<reference checkout> python " + " ".join(sys.argv))
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "tests", "golden")
sys.path.insert(0, ROOT)
sys.path.insert(0, REF)
sys.argv = [sys.argv[0]]
sys.dont_write_bytecode = True

for name, attrs in {
    "einops_exts": dict(check_shape=lambda *a, **k: None, rearrange_many=lambda *a, **k: None),
    "rotary_embedding_torch": dict(RotaryEmbedding=object),
    "video_diffusion_pytorch.text": dict(tokenize=None, bert_embed=None, BERT_MODEL_DIM=768),
}.items():
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    sys.modules[name] = m

from oracle import reference_ops as R  # noqa: E402
from oracle.weights import fill_state_dict, host_noise, synthetic_audio  # noqa: E402
from oracle.metrics import lip_vertex_error  # noqa: E402

import models.hubert as H  # noqa: E402  (reference modules from here on)
import models.wav2vec as W  # noqa: E402

_orig_fwd = H.HubertModel.forward
H.HubertModel.forward = lambda self, x, am=None, **k: _orig_fwd(self, x, None if isinstance(am, str) else am, **k)

torch.manual_seed(0)
torch.set_grad_enabled(False)
N_SAMPLES = 8000  # 0.5 s clips keep the fixtures small; architecture sizes are the real ones
SEED = 7


def set_audio(tiny: bool):
    H.HubertModel.from_pretrained = classmethod(lambda cls, *a, **k: cls(R.audio_encoder_config("hubert", tiny)))
    W.Wav2Vec2Model.from_pretrained = classmethod(lambda cls, *a, **k: cls(R.audio_encoder_config("wav2vec2", tiny)))


def build(preset, tiny=True):
    set_audio(tiny)
    if preset == "vocaset":
        from models.fdm_vocaset import FDM
        from models.vq_vae_vocaset import VQAutoEncoder
        from models.utils.config import vocaset_vq_vae_args as vargs
        from video_diffusion_pytorch.diffusion_BIWI_encoder_decoder import GaussianDiffusion
        fdm = FDM(feature_dim=1024)
    elif preset == "mead":
        from models.fdm_vqvae_mead import FDM
        from models.vq_vae_emotion import VQAutoEncoder
        from utiles.args import vq_vae_args as vargs
        from video_diffusion_pytorch.diffusion_mead_encoder_decoder import GaussianDiffusion
        fdm = FDM(feature_dim=512, vertice_dim=5023 * 3, struct="Dec")
    else:
        from models.fdm import FDM
        from models.vq_vae import VQAutoEncoder
        from models.utils.config import biwi_vq_vae_args as vargs
        from video_diffusion_pytorch.diffusion_BIWI_encoder_decoder import GaussianDiffusion
        fdm = FDM(feature_dim=1024, struct="Dec")
    ae = VQAutoEncoder(vargs())
    diff = GaussianDiffusion(fdm, timesteps=1000, loss_type="l2")
    return fdm.eval(), ae.eval(), diff.eval()


def ref_forward(preset, fdm, audio, t, x, idh, emo):
    tt = torch.full((1,), t, dtype=torch.long)
    if preset == "vocaset":
        return fdm(audio, tt, x, idh)
    if preset == "mead":
        return fdm(audio, tt, x, emo, idh)
    P = R.PRESETS["biwi"]  # harness regroup the BIWI file lacks (SURVEY §8(c) item 6)
    y = fdm(audio, tt, x.reshape(1, x.shape[1] // P["fq"], x.shape[2] * P["fq"]), idh)
    return y.reshape(1, y.shape[1] * P["fq"], y.shape[2] // P["fq"])


def close(a, b, tol, what):
    err = (a - b).abs().max().item()
    ref = b.abs().max().item()
    print(f"  {what}: max|diff| = {err:.3e} (ref max {ref:.3e})")
    assert err <= tol * max(1.0, ref), f"oracle disagrees with the reference on {what}: {err}"


def main():
    os.makedirs(OUT, exist_ok=True)
    # ---- (a) state_dict layout at full size -------------------------------------------------------------
    layout = {}
    for preset in ("vocaset", "mead", "biwi"):
        fdm, ae, diff = build(preset, tiny=False)
        layout[preset] = {
            "diffusion": {k: list(v.shape) for k, v in diff.state_dict().items()},
            "vqvae": {k: list(v.shape) for k, v in ae.state_dict().items()},
        }
        del fdm, ae, diff
    with open(os.path.join(OUT, "state_dict_layout.json"), "w") as f:
        json.dump(layout, f)

    # ---- (b) schedule tables and masks -------------------------------------------------------------------
    _, _, diff = build("mead")
    tabs = R.diffusion_tables(1000)
    table_out = {}
    for k, v in tabs.items():
        assert torch.equal(v, getattr(diff, k)), f"schedule buffer {k} is not bit-exact"
        table_out[k] = v.numpy()
    np.savez_compressed(os.path.join(OUT, "schedule.npz"), **table_out)
    from models.fdm_vocaset import init_biased_mask
    for h, per in ((8, 30), (4, 30), (4, 25)):
        ref_mask = init_biased_mask(n_head=h, max_seq_len=600, period=per)
        assert torch.equal(R.biased_mask(h, 600, per), ref_mask), "closed-form ALiBi mask differs from the reference"
    print("schedule tables and ALiBi masks: bit-exact")

    lip = np.load(os.path.join(REF, "metric", "lip_vertices.npy"))

    # ---- (c) per-preset vectors ---------------------------------------------------------------------------
    for preset in ("vocaset", "mead", "biwi"):
        print(f"[{preset}]")
        P = R.PRESETS[preset]
        fdm, ae, diff = build(preset)
        sd = fill_state_dict(diff.state_dict(), SEED)
        diff.load_state_dict(sd)
        aesd = fill_state_dict(ae.state_dict(), SEED, codebook="reference")
        ae.load_state_dict(aesd)
        fsd = {k[len("denoise_fn."):]: v for k, v in sd.items() if k.startswith("denoise_fn.")}
        audio = synthetic_audio(0, N_SAMPLES)[None]
        hidden = fdm.audio_encoder(audio).last_hidden_state
        hid_o = R.audio_encode(fdm.audio_encoder, audio[0])
        close(hid_o, hidden[0], 1e-5, "audio encoder")
        T = hidden.shape[1] // (2 if P["pair"] else 1)
        idh = torch.eye(P["n_id"])[1][None]
        emo = torch.eye(7)[4][None] if P["emotion"] else None
        x = host_noise(99, 0, 1000, (1, T * P["fq"], P["zdim"]))
        g = {"audio_hidden": hidden[0].numpy(), "x_T": x[0].numpy(), "T": np.int64(T)}
        for t in (999, 500, 0):
            y = ref_forward(preset, fdm, audio, t, x, idh, emo)
            yo = R.fdm_forward(fsd, preset, hidden[0], t, x[0], idh, emo)
            close(yo, y[0], 2e-5, f"x0_hat(t={t})")
            g[f"x0_t{t}"] = y[0].numpy()
        # short ancestral chain through the reference's own p_sample with injected noise
        steps = [999, 998, 997, 2, 1, 0]
        cur = {"t": None}
        real_randn_like = torch.randn_like
        torch.randn_like = lambda z, **k: host_noise(99, 0, cur["t"], tuple(z.shape))
        xr = x.clone()
        try:
            for t in steps:
                cur["t"] = t
                conds = (audio, emo, idh) if preset == "mead" else (audio, idh)
                if preset == "biwi":
                    xx = diff.p_sample(xr.reshape(1, T, -1), torch.full((1,), t, dtype=torch.long), *conds)
                    xr = xx.reshape(1, T * P["fq"], P["zdim"])
                else:
                    xr = diff.p_sample(xr, torch.full((1,), t, dtype=torch.long), *conds)
        finally:
            torch.randn_like = real_randn_like
        xo = R.p_sample_loop(tabs, lambda z, t: R.fdm_forward(fsd, preset, hidden[0], t, z, idh, emo), x[0],
                             lambda t: host_noise(99, 0, t, (1, T * P["fq"], P["zdim"]))[0], steps=steps)
        close(xo, xr[0], 2e-5, "6-step p_sample chain")
        g["chain_steps"] = np.array(steps)
        g["chain_out"] = xr[0].numpy()
        # DDIM (the sampler the shipped VOCASET / BIWI scripts call); x_T injected through torch.randn
        if preset != "mead":
            real_randn = torch.randn
            n_ddim = 6
            try:
                if preset == "biwi":
                    torch.randn = lambda *a, **k: x.reshape(1, T, -1).clone()
                    dd = diff.ddim_sample(audio, (1, T, P["d"]), idh, n_ddim).reshape(1, T * P["fq"], P["zdim"])
                else:
                    torch.randn = lambda *a, **k: x.clone()
                    dd = diff.ddim_sample(audio, tuple(x.shape), idh, n_ddim)
            finally:
                torch.randn = real_randn
            ddo = R.ddim_sample(tabs, lambda z, t: R.fdm_forward(fsd, preset, hidden[0], t, z, idh, emo), x[0], n_ddim)
            close(ddo, dd[0], 2e-5, "6-step ddim_sample")
            g["ddim_steps"] = np.int64(n_ddim)
            g["ddim_out"] = dd[0].numpy()
        # quantise + decode
        emo_pos = int(torch.argmax(emo)) if P["emotion"] else None
        for cb_kind in ("reference", "normal"):
            ae.load_state_dict(fill_state_dict(ae.state_dict(), SEED, codebook=cb_kind))
            cbw = ae.quantize.embedding.weight
            zq, _, (_, _, idx) = ae.quant(xr, emo) if P["emotion"] else ae.quant(xr)
            idx_o, zq_o, margin = R.vq_quantize(xr[0], cbw, emo_pos)
            mism = idx_o != idx[:, 0]
            print(f"  VQ[{cb_kind}]: {int(mism.sum())}/{idx.numel()} rows differ from torch's BLAS-order argmin; "
                  f"largest margin among them {float(margin[mism].max()) if mism.any() else 0.0:.3e}")
            assert float(margin[mism].max() if mism.any() else 0.0) < 1e-5, "oracle argmin differs beyond a rounding tie"
            g[f"vq_idx_{cb_kind}"] = idx[:, 0].numpy()
            g[f"vq_margin_{cb_kind}"] = margin.numpy()
            verts = ae.decode(zq)
            vo = R.vq_decode({k: v for k, v in ae.state_dict().items()}, preset, zq[0])
            close(vo, verts[0], 2e-5, f"decode[{cb_kind}]")
            cols = np.arange(0, verts.shape[-1], 16)
            g[f"verts_cols_{cb_kind}"] = verts[0][:, cols].numpy()
            if verts.shape[-1] == 15069:
                g[f"lve_{cb_kind}"] = np.float64(lip_vertex_error(np.zeros_like(verts[0].numpy()), verts[0].numpy(), lip))
        np.savez_compressed(os.path.join(OUT, f"{preset}.npz"), **g)
        del fdm, ae, diff

    # ---- (d) classifier-free-guidance combine (only the formula is pinned by the reference) ---------------
    from utiles.classifierfree import ClassifierFreeSampleModel
    a, b = torch.randn(1, 24, 64), torch.randn(1, 24, 64)

    class Stub(torch.nn.Module):
        def forward(self, audio, t, x, one_hot, uncond, train=False):
            return b if uncond else a
    out = ClassifierFreeSampleModel(Stub(), level=2.5)(torch.zeros(1, 8), None, torch.zeros(1, 24, 64), None)
    got = R.cfg_forward(lambda oh: a[0] if oh.abs().sum() > 0 else b[0], torch.ones(1, 3), 2.5)
    assert torch.equal(out[0], got), "CFG combine differs from utiles/classifierfree.py"
    np.savez_compressed(os.path.join(OUT, "cfg.npz"), cond=a.numpy(), uncond=b.numpy(), out=out.numpy())
    np.save(os.path.join(OUT, "lip_vertices.npy"), lip)
    print("golden fixtures written to", OUT)


if __name__ == "__main__":
    main()
