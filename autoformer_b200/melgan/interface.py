"""``MelVocoder`` with the reference's surface (melgan/interface.py:23-53), running on the GPU kernels.

``inverse(mel)`` is the conversion path's vocoder call (conversion.ipynb cell 14: ``E.get_wavs(mel.transpose(2, 1))``).
``__call__`` (audio -> mel) runs ``Audio2Mel`` on the same kernel library (melgan/modules.py:26-69, SURVEY.md 8f.4)."""
import os

import torch

from .modules import Audio2Mel, Generator


def get_default_device():
    return "cuda"


class MelVocoder:
    def __init__(self, device=get_default_device(), model_name="multi_speaker", state_dict=None):
        netG = Generator(80, 32, 3)
        if state_dict is None:
            path = f"{model_name}.pt"
            if not os.path.exists(path):
                raise FileNotFoundError(f"{path} not found (the reference loads it the same way, interface.py:29)")
            state_dict = torch.load(path, map_location="cpu")
        netG.load_state_dict(state_dict)
        self.fft = Audio2Mel().to(device)
        self.mel2wav = netG.to(device).eval()
        self.device = device

    def __call__(self, audio):
        """audio (B, L) -> log-mel (B, 80, L // 256)   (interface.py:33-41)."""
        return self.fft(audio.unsqueeze(1).to(self.device))

    def inverse(self, mel, lengths=None):
        """mel (B, 80, T) -> waveform (B, 256 T).  lengths: a zero-padded batch of utterances of lengths[b] frames
        (Generator.forward); samples past 256 lengths[b] are 0."""
        with torch.no_grad():
            if lengths is None:
                return self.mel2wav(mel.to(self.device)).squeeze(1)
            return self.mel2wav(mel.to(self.device), lengths=lengths).squeeze(1)
