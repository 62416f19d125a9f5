# Stand-in for samples/sample_diffusion_vocaset.py of the original Face-Diffusion-Model project: the imports that script makes, as recorded in
# INTEGRATION.md section 1 and SURVEY.md sections 3 and 8(b). Only this import block is part of the fixture.
import os
import sys

import numpy as np
import torch

sys.path.append(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))  # the checkout's root
from datasets.data_loader_vocaset import get_dataloaders
from models.fdm_vocaset import FDM
from models.hubert import HubertModel
from models.utils.config import vocaset_vq_vae_args
from models.vq_vae_vocaset import VQAutoEncoder
from video_diffusion_pytorch.diffusion_BIWI_encoder_decoder import GaussianDiffusion


def main():
    raise SystemExit("stand-in: import block only")
