"""em_sample.m:1-104 -- the legacy file-output driver (RUN_1_emsample.m:38-47), on top of the C ABI.

    em_sample(parameters_filename, initial_output_filename=..., transition_output_filename=...,
              num_initial_samples=100, num_transition_samples=60, start=None,
              isOverwriteZeroBoundaries=False, idxZeroBoundaries=(1, 2, 3), rng_seed=42)

Writes the same two text files: `initial.txt` ("id <labels>" header, one row `id v1 ... vn` per sample,
em_sample.m:59-66,88-92) and `transition.txt` ("initial_id t <labels of the (t+1) variables>" header, one row
`id t x_dyn...` per sample and second, :68-74,94-100), numbers formatted with C's %g like fprintf.
The samples come from emb_sample_tracks (dense compact output: column c is `samples(:, c+1)` of
events2samples.m) and stay on the device, where emb_format_em_sample formats them; only the text crosses PCIe.
`device` (default: the current CUDA device) runs both.  `parms.prior = 'constant'` (em_sample.m:50) is an error in
the reference at HEAD (EncounterModel.m:194-203 accepts only numbers and 'dbe', SURVEY F8); the intended
zero prior is used.  The random stream is the keyed Philox stream with seed `rng_seed`, not MATLAB's twister."""
from __future__ import annotations

from .model import EncounterModel


def em_sample(parameters_filename: str, initial_output_filename: str, transition_output_filename: str,
              num_initial_samples: int = 100, num_transition_samples: int = 60, start=None,
              isOverwriteZeroBoundaries: bool = False, idxZeroBoundaries=(1, 2, 3), rng_seed: int = 42,
              device=None, chunk: int = 1 << 16) -> None:
    parms = EncounterModel(parameters_filename, idxZeroBoundaries=idxZeroBoundaries,
                           isOverwriteZeroBoundaries=isOverwriteZeroBoundaries)
    if start is not None and len(start):
        parms.start = list(start)                                        # em_sample.m:53-55
    n, T = int(num_initial_samples), int(num_transition_samples)
    import torch
    dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    with open(initial_output_filename, "wb") as fi, open(transition_output_filename, "wb") as ft:
        fi.write(("id " + "".join("%s " % l for l in parms.labels_initial) + "\n").encode("utf-8"))                # :59-66
        ft.write(("initial_id t " + "".join("%s " % parms.labels_transition[int(k) - 1]
                                            for k in parms.temporal_map[:, 1]) + "\n").encode("utf-8"))           # :68-74
        for first in range(0, n, chunk):
            m = min(chunk, n - first)
            res = parms.sample_tracks(m, T, seed=rng_seed, first_sample=first, device=dev, want_bins=False)
            text_i, _, text_t, _ = parms.format_em_sample(res, first_id=first + 1)                            # :88-100
            fi.write(text_i.cpu().numpy().tobytes())
            ft.write(text_t.cpu().numpy().tobytes())
