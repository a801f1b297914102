"""Run-to-run reproducibility of the tensor-core modes at the bench batch (8192 x 1 s clips, res15): how many logits
differ between repeated launches on identical inputs, and by how much.  Usage: python tools/determinism_probe.py [precision ...]"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import honk2_b200  # noqa: E402
from honk2_b200 import AudioProcessor, synth  # noqa: E402


def main():
    dev = torch.device("cuda", 0)
    ap = AudioProcessor()
    w = torch.from_numpy(synth.broadband(8192, seed=11)).to(dev)
    feats = ap.compute_mfccs_batch(w)
    for prec in (sys.argv[1:] or ["bf16", "bf16x3"]):
        m = honk2_b200.build_model("res15", precision=prec)
        synth.harden_(m.state_dict())
        m = m.to(dev)
        with torch.no_grad():
            ys = [m(feats).clone() for _ in range(4)]
        scale = float(ys[0].abs().max())
        for k in range(1, 4):
            d = (ys[k] - ys[0]).abs()
            print(f"{prec}: run {k} vs run 0: {int((d > 0).sum())} of {d.numel()} logits differ, max |diff| = "
                  f"{float(d.max()):.3e} ({float(d.max()) / scale:.2e} of the logit scale), rows affected "
                  f"{int((d.amax(1) > 0).sum())}")


if __name__ == "__main__":
    main()
