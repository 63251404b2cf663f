"""Writer / reader of the reference's on-disk token shards (the data format on the output side of the RVQ encode path).

Format (utility_scripts/dump_tokens/dump_tokens.py:217-251): one `torch.save`d dict per file `{rank}_{index}.pt`,
    utterance id -> {"acoustic_codes": [12, L] integer tensor, "semantic_codes": [L] integer tensor,
                     optional "transcription", "no_punc_transcription", "transcription_bytes", "no_punc_transcription_bytes"}
with a new file started every `max_files_per_output_file` utterances (counted in whole batches) and a last partial file.
Readers (edm_tts/datasets/codes_dataset.py:68-83, text_speech_codes_dataset.py:70-98) transpose the acoustic codes to
[L, 12] and cast to int16, so the codes are stored as int16 here as well (values < 1024).
"""
from __future__ import annotations

import glob
import os

import torch

OPTIONAL_KEYS = ("transcription", "no_punc_transcription", "transcription_bytes", "no_punc_transcription_bytes")


class TokenShardWriter:
    """Accumulates utterances of one rank and writes `{rank}_{index}.pt` files like dump_tokens.py does.

        w = TokenShardWriter(out_dir, rank, max_files_per_output_file=10000)
        w.add_batch(ids, acoustic_codes [B, 12, T], semantic_codes [B, T], code_lengths, transcriptions=...)
        w.close()
    """

    def __init__(self, output_dir: str, rank: int = 0, max_files_per_output_file: int = 10000, dtype=torch.int16):
        self.output_dir, self.rank, self.max_items, self.dtype = output_dir, int(rank), int(max_files_per_output_file), dtype
        os.makedirs(output_dir, exist_ok=True)
        self._items: dict = {}
        self._index = 0
        self._counter = 0
        self.files: list[str] = []

    def _path(self) -> str:
        return os.path.join(self.output_dir, f"{self.rank}_{self._index}.pt")

    def add_batch(self, ids, acoustic_codes, semantic_codes, code_lengths=None, **optional):
        """One tokenizer batch: padded tensors acoustic_codes [B, n, T] / semantic_codes [B, T], whose code_lengths[i] trims the
        padded tail (dump_tokens.py:201-222), or per-utterance lists [n, T_i] / [T_i] (e.g. what DAC.encode_to_codes_batch returns),
        which need no code_lengths. Optional per-utterance lists are stored under the reference's singular key names when given
        (plural keyword -> singular key)."""
        B = len(ids)
        lists = isinstance(acoustic_codes, (list, tuple))
        if lists != isinstance(semantic_codes, (list, tuple)):
            raise ValueError("acoustic_codes and semantic_codes must both be lists or both be tensors")
        if len(acoustic_codes) != B or len(semantic_codes) != B:
            raise ValueError("ids, acoustic_codes and semantic_codes must agree on the batch size")
        if lists:
            if any(a.dim() != 2 or s.dim() != 1 or a.shape[-1] != s.shape[-1] for a, s in zip(acoustic_codes, semantic_codes)):
                raise ValueError("every utterance needs acoustic codes [n, T_i] and semantic codes [T_i] of the same T_i")
            ac = [a.detach().to("cpu", self.dtype) for a in acoustic_codes]
            sc = [s.detach().to("cpu", self.dtype) for s in semantic_codes]
        else:
            if acoustic_codes.shape[-1] != semantic_codes.shape[-1]:
                raise ValueError("acoustic and semantic codes must have the same number of frames")  # audio_tokenizer.py:56-57
            ac = acoustic_codes.detach().to("cpu", self.dtype)
            sc = semantic_codes.detach().to("cpu", self.dtype)
        for i, name in enumerate(ids):
            n = int(code_lengths[i]) if code_lengths is not None else ac[i].shape[-1]
            item = {"acoustic_codes": ac[i][:, :n].clone(), "semantic_codes": sc[i][:n].clone()}
            for key in OPTIONAL_KEYS:
                vals = optional.get(key + "s", optional.get(key))
                if vals is not None:
                    item[key] = vals[i]
            self._items[name] = item
        self._counter += B
        if self._counter >= self.max_items:
            self._flush()

    def _flush(self):
        if not self._items:
            return
        path = self._path()
        torch.save(self._items, path)
        self.files.append(path)
        self._items = {}
        self._index += 1
        self._counter = 0

    def close(self) -> list[str]:
        self._flush()
        return self.files


def read_token_shards(data_dir: str):
    """Yields (example id, {"id", "length", "acoustic_tokens" [L, 12] int16, "semantic_tokens" [L, 1] int16}) exactly as the
    reference's CodesDataset._generate_examples does (codes_dataset.py:68-83)."""
    for path in sorted(glob.glob(os.path.join(data_dir, "**", "*.pt"), recursive=True)):
        id_ = os.path.basename(path).replace(".pt", "")
        data = torch.load(path, map_location="cpu")
        for i, (_, v) in enumerate(data.items()):
            acoustic = v["acoustic_codes"].transpose(0, 1).to(torch.int16)
            semantic = v["semantic_codes"][..., None].to(torch.int16)
            yield f"{id_}_{i}", {"id": f"{id_}_{i}", "length": acoustic.shape[0], "acoustic_tokens": acoustic, "semantic_tokens": semantic}
