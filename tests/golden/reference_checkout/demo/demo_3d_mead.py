# Stand-in for demo/demo_3d_mead.py of the original Face-Diffusion-Model project: the imports that script makes, as recorded in
# INTEGRATION.md section 1 and SURVEY.md sections 3 and 8(b). Only this import block is part of the fixture.
import os
import sys

import numpy as np
import torch

sys.path.append(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))  # the checkout's root
import librosa
from transformers import Wav2Vec2Processor
from models.fdm_vqvae_mead import FDM
from models.hubert import HubertModel
from models.vq_vae_emotion import VQAutoEncoder
from utiles.args import vq_vae_args
from utiles.flame_utils import torch2mesh
from video_diffusion_pytorch.diffusion_mead_encoder_decoder import GaussianDiffusion, Unet3D


def main():
    raise SystemExit("stand-in: import block only")
