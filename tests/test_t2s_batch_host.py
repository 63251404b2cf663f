"""CPU checks of the host packing behind TextToSemanticWLen.infer_batch: edm_tts_b200/varlen.py with no prompt rows (P = 0) and one
token per position (Q = 1), as the text-to-semantic batch uses it."""
import torch

from edm_tts_b200 import varlen


def test_plan_without_prompts_chunks_in_order():
    lengths = list(range(1, 140))
    chunks = varlen.plan(lengths, [0] * len(lengths), 64, batch_offset=7)
    assert [(c.start, c.stop) for c in chunks] == [(0, 64), (64, 128), (128, 139)]
    assert [c.batch_offset for c in chunks] == [7, 71, 135]
    assert [c.t0 for c in chunks] == [0, sum(lengths[:64]), sum(lengths[:128])]
    assert all(set(c.P) == {0} for c in chunks)


def test_split_blocks_gives_per_utterance_token_views():
    lengths = [3, 1, 5]
    out = torch.arange(sum(lengths))
    views = [b[0] for b in varlen.split_blocks(out, lengths, 1)]
    assert [v.tolist() for v in views] == [[0, 1, 2], [3], [4, 5, 6, 7, 8]]
    views[1][0] = -1  # views of the one packed output, not copies
    assert out[3] == -1
