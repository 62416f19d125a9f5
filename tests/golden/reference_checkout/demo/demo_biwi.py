# Stand-in for demo/demo_biwi.py of the original Face-Diffusion-Model project: the imports that script makes, as recorded in
# INTEGRATION.md section 1 and SURVEY.md sections 3 and 8(b). Only this import block is part of the fixture.
import os
import sys

import numpy as np
import torch

sys.path.append(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))  # the checkout's root
import librosa
from transformers import Wav2Vec2Processor
from models.fdm import FDM
from models.utils.config import biwi_vq_vae_args
from models.vq_vae import VQAutoEncoder
from models.wav2vec import Wav2Vec2Model
from video_diffusion_pytorch.diffusion_BIWI_encoder_decoder import GaussianDiffusion


def main():
    raise SystemExit("stand-in: import block only")
