# Stand-in for samples/sample_mead_vqvae.py of the original Face-Diffusion-Model project: the imports that script makes, as recorded in
# INTEGRATION.md section 1 and SURVEY.md sections 3 and 8(b). Only this import block is part of the fixture.
import os
import sys

import numpy as np
import torch

sys.path.append(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))  # the checkout's root
from datasets.data_loader_mead_vqvae import get_dataloaders
from models.vq_vae_emotion import VQAutoEncoder
from utiles.args import vq_vae_args


def main():
    raise SystemExit("stand-in: import block only")
