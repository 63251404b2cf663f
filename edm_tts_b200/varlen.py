"""Host-side layout of a variable-length S2A batch (plain Python, no GPU): where each utterance sits in the packed buffers of
edm_s2a_bind_varlen, how a long list is cut into chunks, and the per-utterance views of the packed output.

Utterance i has T_i target and P_i prompt frames. Packed buffers hold the utterances back to back: per-frame data of utterance i
starts at cu_t[i] (targets) or cu_p[i] (prompt), a per-utterance [Q, T_i] block at Q * cu_t[i]. With equal lengths this is the
[B, ...] layout of a uniform batch.
"""
from __future__ import annotations

from dataclasses import dataclass


def offsets(lengths) -> list[int]:
    """[0, l0, l0 + l1, ...]: the start of every item in a packed buffer, and the total at the end."""
    out = [0]
    for n in lengths:
        out.append(out[-1] + int(n))
    return out


@dataclass(frozen=True)
class Chunk:
    """Utterances [start, stop) of the caller's list, decoded by one bound workspace."""
    start: int
    stop: int
    batch_offset: int   # global index of the chunk's first utterance (Philox counters)
    T: tuple            # target frames per utterance
    P: tuple            # prompt frames per utterance
    t0: int             # first target frame of the chunk in the whole packed batch


def plan(T, P, max_chunk: int, batch_offset: int = 0) -> list[Chunk]:
    """Cut the list into chunks of at most max_chunk utterances, in the given order."""
    if len(T) != len(P):
        raise ValueError(f"{len(T)} target lengths but {len(P)} prompt lengths")
    cu_t = offsets(T)
    return [Chunk(s, min(len(T), s + max_chunk), int(batch_offset) + s, tuple(T[s:s + max_chunk]), tuple(P[s:s + max_chunk]), cu_t[s])
            for s in range(0, len(T), max_chunk)]


def split_blocks(packed, T, Q: int) -> list:
    """Views [Q, T_i] of a flat packed buffer of per-utterance [Q, T_i] blocks."""
    cu = offsets(T)
    return [packed[Q * cu[i]:Q * cu[i + 1]].view(Q, T[i]) for i in range(len(T))]
