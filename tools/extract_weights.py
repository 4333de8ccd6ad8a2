#!/usr/bin/env python
"""Extract the Silero-VAD v6.2.1 parameters from the reference TorchScript archive.

Runs only in the build container (needs /root/reference).  The only trusted weight
source is `src/silero_vad/data/silero_vad.jit` (SURVEY.md F6); its `state_dict()`
holds 30 fp32 tensors (15 per sample-rate branch).

Outputs (raw little-endian fp32, "SVADW001" container, see silero_vad_b200.tuning.write_container):
  silero_vad_b200/data/silero_vad_v6.weights   28 tensors (no STFT bases) - product
  oracle/data/stft_basis.weights                2 tensors (STFT conv bases) - oracle only
"""
import sys
from pathlib import Path

import torch

REPO = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(REPO))
from silero_vad_b200.tuning import write_container  # noqa: E402  (the one SVADW001 writer)
JIT = Path("/root/reference/src/silero_vad/data/silero_vad.jit")


def main():
    m = torch.jit.load(str(JIT), map_location="cpu").eval()
    sd = m.state_dict()
    assert len(sd) == 30, len(sd)
    prod, basis = [], []
    for k, v in sd.items():
        assert v.dtype == torch.float32
        (basis if "forward_basis_buffer" in k else prod).append((k, v))
    write_container(REPO / "silero_vad_b200/data/silero_vad_v6.weights", prod)
    write_container(REPO / "oracle/data/stft_basis.weights", basis)
    for name, lst in (("product", prod), ("oracle-basis", basis)):
        print(name, len(lst), "tensors", sum(t.numel() for _, t in lst) * 4, "bytes")


if __name__ == "__main__":
    sys.exit(main())
