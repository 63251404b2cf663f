"""Host-side layout of variable-length batches (plain Python, no GPU): where each utterance sits in the packed buffers, how a long
list is cut into chunks, and the per-utterance views of the packed output.

S2A (edm_s2a_bind_varlen): utterance i has T_i target and P_i prompt frames. Packed buffers hold the utterances back to back:
per-frame data of utterance i starts at cu_t[i] (targets) or cu_p[i] (prompt), a per-utterance [Q, T_i] block at Q * cu_t[i]. With
equal lengths this is the [B, ...] layout of a uniform batch.

S2A infilling (edm_s2a_bind_masked): the same with the known (prompt) frames anywhere in their utterance, see infill_split.
Text-to-semantic infilling (edm_t2s_begin_masked): a text-to-semantic batch with some speech positions known, see t2s_infill_split.

DAC decoder (DACDecoder.forward_batch): the utterances are packed along time with zero gap rows between them, see dac_pack.
DAC encoder (DACEncoder.forward_batch): the same idea for the downsampling stack, see enc_pack.
"""
from __future__ import annotations

import math
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


def cut(n: int, rows, limit: int) -> list[tuple[int, int]]:
    """Cut items [0, n), in order, into ranges [s, e) whose packed rows rows(s, e) stay within limit; an item that alone exceeds the
    limit gets a range of its own."""
    out, s = [], 0
    while s < n:
        e = s + 1
        while e < n and rows(s, e + 1) <= limit:
            e += 1
        out.append((s, e))
        s = e
    return out


def split_blocks(packed, T, Q: int) -> list:
    """Views [Q, T_i] of a flat packed buffer of per-utterance [Q, T_i] blocks."""
    cu = offsets(T)
    return [packed[Q * cu[i]:Q * cu[i + 1]].view(Q, T[i]) for i in range(len(T))]


# ---------------------------------------------------------------------------------------------------------------------------------
# S2A infilling (edm_s2a_bind_masked): utterance i has N_i frames, T_i >= 1 of them marked to regenerate (targets), the other
# P_i = N_i - T_i known. Per-target data is packed as a varlen batch with T_i targets, per-known data as its prompt of P_i frames, both
# in time order; the encoder rows keep the utterance's own frame order.


@dataclass(frozen=True)
class Infill:
    """An infill batch split into what the masked bind takes: per utterance the frame count, the target / known counts, the
    semantic tokens of the targets and of the known frames, the codes [q, P_i] of the known frames and the bool target mask."""
    N: tuple
    T: tuple
    P: tuple
    sem_target: list
    sem_known: list
    codes_known: list
    target: list


def infill_split(semantic_tokens, acoustic_tokens, regenerate, num_codes: int, num_semantic: int, max_levels: int = 12) -> Infill:
    """Checks an infill batch (lists of semantic tokens [N_i], acoustic codes [q, N_i] with one q in [1, max_levels], bool masks [N_i]
    of the frames to regenerate) and splits it into targets and known frames. Malformed lists or shapes and an utterance with no frame
    to regenerate raise ValueError; a semantic token or a known frame's code out of range raises IndexError (the codes at regenerated
    frames are ignored)."""
    import torch

    lists = (semantic_tokens, acoustic_tokens, regenerate)
    if any(not isinstance(x, (list, tuple)) for x in lists) or len(semantic_tokens) == 0:
        raise ValueError("semantic_tokens, acoustic_tokens and regenerate must be non-empty lists")
    n = len(semantic_tokens)
    if len(acoustic_tokens) != n or len(regenerate) != n:
        raise ValueError(f"{n} semantic token lists, {len(acoustic_tokens)} acoustic and {len(regenerate)} regenerate masks")
    if any(not torch.is_tensor(x) for lst in lists for x in lst):
        raise ValueError("every entry must be a tensor")
    q = int(acoustic_tokens[0].shape[0]) if acoustic_tokens[0].dim() == 2 else -1
    N, T = [], []
    for i, (st, ac, rg) in enumerate(zip(*lists)):
        if st.dim() != 1 or ac.dim() != 2 or rg.dim() != 1:
            raise ValueError(f"utterance {i}: expected semantic [N], acoustic [q, N] and regenerate [N] tensors")
        if int(ac.shape[0]) != q or not 1 <= q <= max_levels:
            raise ValueError(f"utterance {i}: every acoustic entry needs the same number of levels q in [1, {max_levels}]")
        if ac.shape[1] != st.shape[0] or rg.shape[0] != st.shape[0]:
            raise ValueError(f"utterance {i}: {st.shape[0]} semantic tokens, {ac.shape[1]} acoustic frames, {rg.shape[0]} mask entries")
        if rg.dtype != torch.bool:
            raise ValueError(f"regenerate[{i}] must be a bool tensor")
        t = int(rg.sum())
        if t < 1:
            raise ValueError(f"utterance {i} has no frame to regenerate")
        N.append(int(st.shape[0]))
        T.append(t)
    sem_t, sem_k, codes_k, tgt = [], [], [], []
    for i, (st, ac, rg) in enumerate(zip(*lists)):
        rg = rg.to(st.device)
        if st.numel() and (int(st.min()) < 0 or int(st.max()) >= num_semantic):
            raise IndexError(f"semantic_tokens[{i}]: index out of range [0, {num_semantic})")
        known = ac[:, ~rg.to(ac.device)]
        if known.numel() and (int(known.min()) < 0 or int(known.max()) >= num_codes):
            raise IndexError(f"acoustic_tokens[{i}]: a known frame's code is out of range [0, {num_codes})")
        sem_t.append(st[rg])
        sem_k.append(st[~rg])
        codes_k.append(known)
        tgt.append(rg)
    return Infill(tuple(N), tuple(T), tuple(a - b for a, b in zip(N, T)), sem_t, sem_k, codes_k, tgt)


def infill_rows(target) -> tuple[list[int], list[int]]:
    """Row maps of a masked bind for the bool masks `target` [N_i] of its utterances (what edm_s2a_bind_masked builds on the host):
    tgt_enc[r] = packed encoder row of packed target row r; enc_slot[row] = target index t inside the utterance, or -1 - k for its
    k-th known frame."""
    tgt_enc, enc_slot, row = [], [], 0
    for m in target:
        t = k = 0
        for v in (bool(x) for x in m):
            if v:
                tgt_enc.append(row)
                enc_slot.append(t)
                t += 1
            else:
                enc_slot.append(-1 - k)
                k += 1
            row += 1
    return tgt_enc, enc_slot


# ---------------------------------------------------------------------------------------------------------------------------------
# Text-to-semantic infilling (edm_t2s_begin_masked): utterance i is a transcript of n_text_i tokens and N_i speech positions, T_i >= 1
# of them regenerated, the others known. Its sequence has L_i = n_text_i + N_i + 4 rows, speech position k at row n_text_i + 3 + k.
# Per-position data (known tokens, regenerate flags) is packed [sum N_i], the regenerated tokens [sum T_i], both in time order.


@dataclass(frozen=True)
class T2sInfill:
    """A checked text-to-semantic infill batch: per utterance the speech positions N_i and the regenerated ones T_i; the packed
    semantic tokens [sum N_i] (int64, on the tokens' device, 0 at regenerated positions) and regenerate flags [sum N_i] (uint8, host)."""
    N: tuple
    T: tuple
    known: object
    regenerate: object


def t2s_infill_split(n_text, semantic_tokens, regenerate, num_semantic: int, max_positions: int) -> T2sInfill:
    """Checks a text-to-semantic infill batch (transcript lengths n_text_i, semantic tokens [N_i], bool masks [N_i] of the positions
    to regenerate) and packs it. Raises ValueError naming the utterance when the lists differ in length, a mask and its tokens differ
    in length, an utterance has nothing to regenerate, a known token lies outside [0, num_semantic) (values at regenerated positions
    are ignored), or L_i = n_text_i + N_i + 4 exceeds max_positions."""
    import torch

    if not isinstance(semantic_tokens, (list, tuple)) or not isinstance(regenerate, (list, tuple)) or len(semantic_tokens) == 0:
        raise ValueError("semantic_tokens and regenerate must be non-empty lists")
    n = len(semantic_tokens)
    if len(regenerate) != n or len(n_text) != n:
        raise ValueError(f"{len(n_text)} texts, {n} semantic token lists and {len(regenerate)} regenerate masks")
    N, T = [], []
    for i, (st, rg) in enumerate(zip(semantic_tokens, regenerate)):
        if not torch.is_tensor(st) or not torch.is_tensor(rg) or st.dim() != 1 or rg.dim() != 1:
            raise ValueError(f"utterance {i}: expected semantic_tokens [N] and regenerate [N] tensors")
        if rg.dtype != torch.bool:
            raise ValueError(f"utterance {i}: regenerate must be a bool tensor")
        if rg.shape[0] != st.shape[0]:
            raise ValueError(f"utterance {i}: {st.shape[0]} semantic tokens but {rg.shape[0]} regenerate entries")
        t = int(rg.sum())
        if t < 1:
            raise ValueError(f"utterance {i} has no speech position to regenerate")
        L = int(n_text[i]) + st.shape[0] + 4
        if L > max_positions:
            raise ValueError(f"utterance {i}: sequence of {L} tokens exceeds max_positions={max_positions}")
        N.append(int(st.shape[0]))
        T.append(t)
    dev = semantic_tokens[0].device
    regen = torch.cat([r.cpu() for r in regenerate])
    known = torch.cat([s.to(dev, torch.int64) for s in semantic_tokens]).masked_fill(regen.to(dev), 0)
    lo, hi = torch.aminmax(known)
    if int(lo) < 0 or int(hi) >= num_semantic:
        cu = offsets(N)
        for i in range(n):
            seg = known[cu[i]:cu[i + 1]]
            if int(seg.min()) < 0 or int(seg.max()) >= num_semantic:
                raise ValueError(f"utterance {i}: a known semantic token is out of range [0, {num_semantic})")
    return T2sInfill(tuple(N), tuple(T), known, regen.to(torch.uint8))


def t2s_infill_maps(n_text, regenerate) -> tuple[list[int], list[int]]:
    """The two maps edm_t2s_begin_masked builds on the host for masks `regenerate` [N_i] of sequences with n_text_i text tokens:
    regen_slot[cu_N[i] + k] = index of speech position k of utterance i among the regenerated positions of the batch, or -1 when it
    is known; regen_row[j] = packed row of regenerated position j."""
    regen_slot, regen_row, row0, j = [], [], 0, 0
    for nt, m in zip(n_text, regenerate):
        for k, v in enumerate(bool(x) for x in m):
            regen_slot.append(j if v else -1)
            if v:
                regen_row.append(row0 + int(nt) + 3 + k)
                j += 1
        row0 += int(nt) + len(m) + 4
    return regen_slot, regen_row


# ---------------------------------------------------------------------------------------------------------------------------------
# DAC decoder batches: utterances packed along time with zero gap rows between them (DESIGN §4a). The conv kernels zero-fill only at
# the two ends of a tensor, so every utterance gets its conv padding from gap rows that are exactly zero when a conv reads them.
# Stage 0 is the latent (and the first conv's output, same rows); stage k follows the k-th transposed conv (stride r_k). Utterance i
# starts at a[k][i] = r_k * a[k-1][i] and has L[k][i] = conv_transpose_length(L[k-1][i], r_k) rows, so the transposed conv's output
# view (out_view[q] -> out[q r + phase - pad]) lands every utterance at its packed place without any new indexing.

DAC_FIRST_READ = 3      # first conv k=7 (reads the latent)
DAC_UNIT_READ = 27      # dilation-9 k=7 conv of the last ResidualUnit of every upsampled stage
DAC_LAST_READ = 3       # last conv k=7
DAC_UP_READ = 1         # transposed conv as a 2-tap conv: x[q - 1], x[q]


def conv_transpose_length(L_in: int, stride: int) -> int:
    """Output length of ConvTranspose1d(kernel 2s, stride s, padding floor(s/2), output_padding s % 2) (decoder.py:15-23)."""
    return (L_in - 1) * stride - 2 * (stride // 2) + 2 * stride + stride % 2


def dac_stage_reads(rates) -> list[int]:
    """Widest one-sided read into each stage's bf16 operand: the first conv and the first transposed conv read stage 0, the
    ResidualUnits, the next transposed conv (or the last conv) read stage k >= 1."""
    K = len(rates)
    return [max(DAC_FIRST_READ, DAC_UP_READ)] + [max(DAC_UNIT_READ, DAC_UP_READ if k < K else DAC_LAST_READ) for k in range(1, K + 1)]


def dac_stage_gaps(g0: int, rates) -> list[int]:
    """Rows between two neighbouring utterances (and after the last one) at each stage, for a latent gap of g0 rows:
    g_k = r_k g_{k-1} - 2 (r_k % 2). The gap in front of the first utterance is prod(r) g0 >= g_k."""
    out = [int(g0)]
    for r in rates:
        out.append(r * out[-1] - 2 * (r % 2))
    return out


def min_gap(stage_gaps, reads) -> int:
    """Smallest gap g >= 1 whose stage gaps stage_gaps(g) cover every stage's widest one-sided read reads[k]."""
    g = 1
    while any(x < n for x, n in zip(stage_gaps(g), reads)):
        g += 1
    return g


def dac_min_gap(rates) -> int:
    """Smallest latent gap G0 whose gaps cover every stage's widest one-sided read."""
    if any(int(r) < 2 for r in rates):
        raise ValueError(f"transposed-conv strides must be >= 2 (output_padding s % 2 < s), got {tuple(rates)}")
    return min_gap(lambda g: dac_stage_gaps(g, rates), dac_stage_reads(rates))


@dataclass(frozen=True)
class DacChunk:
    """Utterances [start, stop) of the caller's list, run through one packed pass. rows[k] packed rows of stage k, starts[k][i] /
    lengths[k][i] where utterance start + i sits in them; t0 is the chunk's first row in the concatenated input (latent frames for
    the decoder, audio samples for the encoder)."""
    start: int
    stop: int
    t0: int
    rows: tuple
    starts: tuple
    lengths: tuple

    def gaps(self, k: int) -> list[tuple[int, int]]:
        """[start, end) row ranges of stage k outside every utterance: exactly the complement of the valid ranges in [0, rows[k])."""
        out, prev = [], 0
        for a, n in zip(self.starts[k], self.lengths[k]):
            out.append((prev, a))
            prev = a + n
        out.append((prev, self.rows[k]))
        return out


def dac_pack(T, rates, g0: int, start: int = 0, t0: int = 0) -> DacChunk:
    """Packed geometry of utterances with T[i] latent frames, laid out as | g0 | T_0 | g0 | T_1 | ... | T_n-1 | g0 |."""
    a, n = [], []
    pos = g0
    for t in T:
        a.append(pos)
        n.append(int(t))
        pos += int(t) + g0
    rows, starts, lengths = [pos], [tuple(a)], [tuple(n)]
    for r in rates:
        rows.append(r * rows[-1])
        starts.append(tuple(r * x for x in starts[-1]))
        lengths.append(tuple(conv_transpose_length(x, r) for x in lengths[-1]))
    return DacChunk(start, start + len(T), t0, tuple(rows), tuple(starts), tuple(lengths))


def dac_plan(T, rates, max_chunk_samples: int) -> list[DacChunk]:
    """Cut the list, in order, into chunks whose packed audio rows (gaps included) stay within max_chunk_samples; an utterance that
    alone exceeds the limit gets a chunk of its own."""
    g0 = dac_min_gap(rates)
    hop = math.prod(rates)
    cu = offsets(T)
    rows = lambda s, e: hop * (g0 * (e - s + 1) + cu[e] - cu[s])               # | g0 | T_s | g0 | ... | T_e-1 | g0 | in audio rows
    return [dac_pack(T[s:e], rates, g0, s, cu[s]) for s, e in cut(len(T), rows, max_chunk_samples)]


# ---------------------------------------------------------------------------------------------------------------------------------
# DAC encoder batches: clips packed along time with zero gap rows, for the downsampling stack (DESIGN §4a). Stage 0 is the audio (and
# the first conv's output, same rows); stage k follows the k-th strided conv (kernel 2s, stride s, padding ceil(s/2)), which reads its
# operand through a [rows / s][s C] view: a clip's output lands at its packed place only if its start is a multiple of s at every stage,
# so in audio rows every clip starts at a multiple of the hop. Clip i takes a slot of ceil(L_i / hop) + G latent frames behind G frames
# in front of the first clip; at stage k (cumulative stride r_k) it starts at a[0][i] / r_k and has the single-path length chain
# L[k][i] = strided_conv_length(L[k-1][i], s_k).

ENC_FIRST_READ = 3      # first conv k=7 (reads the packed audio)
ENC_UNIT_READ = 27      # dilation-9 k=7 conv of the last ResidualUnit of every stage before a strided conv
ENC_LAST_READ = 1       # last conv k=3 (reads the latent)


def strided_conv_length(L_in, stride: int):
    """Output length of Conv1d(kernel 2s, stride s, padding ceil(s/2)) (encoder.py:19-25); works on ints and integer tensors. The
    other convs of the encoder (k=7 pad 3, dilated k=7 pad 3d, k=1, k=3 pad 1) keep the length."""
    return (L_in + 2 * math.ceil(stride / 2) - 2 * stride) // stride + 1


def enc_stage_reads(rates) -> list[int]:
    """Widest one-sided read into each stage's operand: the ResidualUnits and the strided conv (ceil(s/2) rows on either side) read
    stages 0 .. K-1 (the first conv reads the audio at stage 0), the last conv reads the latent (stage K)."""
    return ([max(ENC_FIRST_READ, ENC_UNIT_READ, math.ceil(rates[0] / 2))] + [max(ENC_UNIT_READ, math.ceil(s / 2)) for s in rates[1:]]
            + [ENC_LAST_READ])


def enc_stage_gaps(g: int, rates) -> list[int]:
    """Narrowest gap at each stage for a latent gap of g frames: (hop / r_k) g rows, reached when the clip in front of it is a
    multiple of the hop long (a shorter clip leaves more)."""
    out = [int(g) * math.prod(rates)]
    for s in rates:
        out.append(out[-1] // s)
    return out


def enc_min_gap(rates) -> int:
    """Smallest latent gap G whose gaps cover every stage's widest one-sided read."""
    if not rates or any(int(s) < 2 for s in rates):
        raise ValueError(f"strides must be >= 2 (a stride-1 conv of kernel 2 lengthens the clip into its gap), got {tuple(rates)}")
    return min_gap(lambda g: enc_stage_gaps(g, rates), enc_stage_reads(rates))


def enc_rows(frames: int) -> int:
    """Packed latent rows for `frames` latent frames of gaps and slots: rounded up to a multiple of 8 by lengthening the tail gap, so
    bf16 z rows are 16-byte multiples, as the RVQ's TMA maps read them."""
    return (frames + 7) // 8 * 8


def enc_slot(L_i: int, hop: int, g: int) -> int:
    """Latent frames of clip i's slot: ceil(L_i / hop) frames for the clip, then a gap of g."""
    return -(-int(L_i) // hop) + g


def enc_pack(L, rates, g: int, start: int = 0, t0: int = 0) -> DacChunk:
    """Packed geometry of clips with L[i] audio samples (stage 0 = audio, stage K = latent)."""
    hop = math.prod(rates)
    a, pos = [], g
    for x in L:
        a.append(hop * pos)
        pos += enc_slot(x, hop, g)
    rows, starts, lengths = [hop * enc_rows(pos)], [tuple(a)], [tuple(int(x) for x in L)]
    for s in rates:
        rows.append(rows[-1] // s)
        starts.append(tuple(x // s for x in starts[-1]))
        lengths.append(tuple(strided_conv_length(x, s) for x in lengths[-1]))
    return DacChunk(start, start + len(L), t0, tuple(rows), tuple(starts), tuple(lengths))


def enc_plan(L, rates, max_chunk_samples: int) -> list[DacChunk]:
    """Cut the list, in order, into chunks whose packed audio rows (gaps included) stay within max_chunk_samples; a clip that alone
    exceeds the limit gets a chunk of its own."""
    g = enc_min_gap(rates)
    hop = math.prod(rates)
    cu, cu_slot = offsets(L), offsets(enc_slot(x, hop, g) for x in L)
    rows = lambda s, e: hop * enc_rows(g + cu_slot[e] - cu_slot[s])             # enc_pack's rows[0]
    return [enc_pack(L[s:e], rates, g, s, cu[s]) for s, e in cut(len(L), rows, max_chunk_samples)]
