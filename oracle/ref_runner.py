"""Runs the REAL reference modules on the host cores (TEST / BASELINE INFRASTRUCTURE; never imported by the product).

`bench.py --impl reference` and bench.py's `cpu_baseline` leg time the reference's own PyTorch implementation of the
sampling path. The reference has no packaging (no setup.py / pyproject.toml), so it cannot be pip-installed into
`baseline/_ref`; instead `__graft_entry__.build()`, given a checkout of it in FDM_B200_REFERENCE_DIR, copies the
reference's hot-path packages (models/, utiles/, video_diffusion_pytorch/: the files SURVEY.md section 8(a) cites)
UNMODIFIED into the git-ignored `oracle/_ref/`. This module imports them from there with the harness shims of SURVEY.md
section 8(c) (missing optional modules stubbed, audio encoders built from their configs with random weights,
zero-initialised output layer re-initialised) and drives them exactly as samples/sample_diffusion_*.py do: B = 1, the
audio encoder re-run inside every denoiser call, `diffusion.p_sample` per step. Classifier-free guidance follows
utiles/classifierfree.py:15-21 (two denoiser calls per step, the second with the null condition).

When `oracle/_ref` is absent (build() ran without FDM_B200_REFERENCE_DIR) callers fall back to the oracle port
(oracle/reference_ops.py) and say so (`cpu_baseline.kind == "port"`)."""
import os
import sys
import time
import types

HERE = os.path.dirname(os.path.abspath(__file__))
REF_DIR = os.path.join(HERE, "_ref")
REF_PACKAGES = ("models", "utiles", "video_diffusion_pytorch")


def available() -> bool:
    return all(os.path.isdir(os.path.join(REF_DIR, p)) for p in REF_PACKAGES)


def install_from(src: str) -> bool:
    """Copy the reference's hot-path packages (python files only, unmodified) from the checkout `src` into oracle/_ref."""
    import shutil
    if not os.path.isdir(src):
        return False
    for pkg in REF_PACKAGES:
        dst = os.path.join(REF_DIR, pkg)
        if os.path.isdir(dst):
            shutil.rmtree(dst)
        shutil.copytree(os.path.join(src, pkg), dst, ignore=shutil.ignore_patterns("__pycache__", "*.pyc"))
    return True


def _import_reference():
    """Import the reference modules from oracle/_ref in a way that cannot collide with the drop-in packages of the same
    names: the caller must be a process that has NOT imported face-diffusion-model_b200's `models` (bench.py runs the
    reference in a subprocess)."""
    assert available(), "oracle/_ref is missing: run __graft_entry__.build() with FDM_B200_REFERENCE_DIR set"
    for name in ("models", "utiles", "video_diffusion_pytorch"):
        assert name not in sys.modules, f"{name} already imported: run the reference in its own process"
    sys.path.insert(0, REF_DIR)
    sys.argv = [sys.argv[0]]
    for name, attrs in {
        "einops_exts": dict(check_shape=lambda *a, **k: None, rearrange_many=lambda *a, **k: None),
        "rotary_embedding_torch": dict(RotaryEmbedding=object),
        "video_diffusion_pytorch.text": dict(tokenize=None, bert_embed=None, BERT_MODEL_DIM=768),
    }.items():
        if name not in sys.modules:
            m = types.ModuleType(name)
            m.__dict__.update(attrs)
            sys.modules[name] = m
    from transformers import HubertConfig, Wav2Vec2Config
    import models.hubert as H
    import models.wav2vec as W
    hcfg = HubertConfig(hidden_size=1024, num_hidden_layers=24, num_attention_heads=16, intermediate_size=4096,
                        feat_extract_norm="layer", do_stable_layer_norm=True, conv_bias=True, attn_implementation="eager")
    H.HubertModel.from_pretrained = classmethod(lambda cls, *a, **k: cls(hcfg))
    W.Wav2Vec2Model.from_pretrained = classmethod(lambda cls, *a, **k: cls(Wav2Vec2Config(attn_implementation="eager")))
    orig = H.HubertModel.forward  # models/fdm_vocaset.py:59 passes the dataset name as attention_mask
    H.HubertModel.forward = lambda self, x, am=None, **k: orig(self, x, None if isinstance(am, str) else am, **k)
    return H, W


def build(preset: str):
    """(fdm, autoencoder, diffusion) of the reference, random init (latent_decoder re-initialised: SURVEY section 0)."""
    import torch
    _import_reference()
    torch.manual_seed(0)
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
    torch.nn.init.normal_(fdm.latent_decoder.weight, std=0.02)
    ae = VQAutoEncoder(vargs())
    diff = GaussianDiffusion(fdm, timesteps=1000, loss_type="l2")
    return fdm.eval(), ae.eval(), diff.eval()


def _denoiser(fdm, preset: str, T: int, fq: int, zdim: int, guidance: bool, level: float = 2.5):
    """The reference FDM as GaussianDiffusion.denoise_fn: plus the latent regroup models/fdm.py lacks (SURVEY section 8(c)
    item 6) and, with guidance, utiles/classifierfree.py:15-21 restated as a harness wrapper (the shipped wrapper's call
    signature matches no FDM, item 9): cond pass, null-condition pass, uncond + level * (cond - uncond)."""
    import torch

    class Wrapped(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.model = fdm

        def one(self, audio, t, x, *conds):
            if preset == "biwi":
                return self.model(audio, t, x.reshape(1, T, fq * zdim), *conds).reshape(1, T * fq, zdim)
            return self.model(audio, t, x, *conds)

        def forward(self, audio, t, x, *conds):
            out = self.one(audio, t, x, *conds)
            if not guidance:
                return out
            null = list(conds)
            null[0] = torch.zeros_like(null[0])  # emotion one-hot (mead) / identity one-hot (vocaset, biwi)
            out_u = self.one(audio, t, x, *null)
            return out_u + level * (out - out_u)

    return Wrapped().eval()


def time_sampling(preset: str, seconds: float, n_steps: int, total_steps: int, guidance: bool, threads: int,
                  samples: int = 1, warmup_samples: int = 0, warmup_steps: int = 2):
    """One clip through the reference as its sample scripts run it. A SAMPLE = `n_steps` DDPM steps (t = 998 ...) through
    `diffusion.p_sample` plus quantise + decode, extrapolated to `total_steps`; `warmup_samples` shorter untimed samples
    first. Returns a list of dicts (one per timed sample): fps, frames, s_per_step, quant_decode_s, sample_s, cores."""
    import torch
    torch.set_num_threads(threads)
    fdm, ae, diff = build(preset)
    n = int(16000 * seconds)
    g = torch.Generator(device="cpu").manual_seed(1234)
    audio = torch.randn(1, n, generator=g)
    audio = (audio - audio.mean()) / audio.std()
    if preset == "mead":
        conds = (torch.eye(7)[4][None], torch.eye(25)[0][None])
    elif preset == "vocaset":
        conds = (torch.eye(8)[0][None],)
    else:
        conds = (torch.eye(6)[0][None],)
    fq, zdim, pair = {"vocaset": (16, 64, False), "mead": (8, 64, True), "biwi": (8, 128, True)}[preset]
    with torch.no_grad():
        N = fdm.audio_encoder(audio).last_hidden_state.shape[1]
    T = N // 2 if pair else N
    shape = (1, T * fq, zdim)
    diff.denoise_fn = _denoiser(fdm, preset, T, fq, zdim, guidance)

    def one(steps):
        x = torch.randn(shape)
        t0 = time.perf_counter()
        for i in range(steps):
            x = diff.p_sample(x, torch.full((1,), 998 - i, dtype=torch.long), audio, *conds)
        loop = time.perf_counter() - t0
        t1 = time.perf_counter()
        with torch.no_grad():
            q = ae.quant(x, conds[0]) if preset == "mead" else ae.quant(x)
            v = ae.decode(q[0])
        tail = time.perf_counter() - t1
        assert v.shape[1] == T
        per_step = loop / steps
        return dict(fps=T / (per_step * total_steps + tail), frames=T, s_per_step=per_step, quant_decode_s=tail,
                    sample_s=loop + tail, cores=threads, sampled_steps=steps)

    for _ in range(warmup_samples):
        one(warmup_steps)
    return [one(n_steps) for _ in range(samples)]


if __name__ == "__main__":
    # python oracle/ref_runner.py preset seconds n_steps total_steps guidance threads [samples warmup_samples] -> JSON list
    import json
    a = sys.argv[1:]
    print(json.dumps(time_sampling(a[0], float(a[1]), int(a[2]), int(a[3]), a[4] == "1", int(a[5]),
                                   int(a[6]) if len(a) > 6 else 1, int(a[7]) if len(a) > 7 else 0)))
