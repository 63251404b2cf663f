// Where the sequences of a bound batch live in the row buffers of the decoder (the one place that knows it).
// Sequence s has P_s >= 0 prompt rows followed by T_s >= 1 target rows, N_s = P_s + T_s encoder rows. The sequences are packed
// back to back without padding:
//   encoder rows (x, z, h, qkv, g, ...)   sequence s starts at row cu_n[s]
//   target rows (zt, logits, ids, mask)   sequence s starts at row cu_t[s]
//   per-sequence prompt tokens            sequence s starts at cu_p[s] = cu_n[s] - cu_t[s]  (q levels: q * cu_p[s])
//   [Q, T_s] blocks (codes, coarse ids)   sequence s starts at Q * cu_t[s]
// A uniform batch (every sequence N rows, T of them targets) is the same layout with cu_n[s] = s N and cu_t[s] = s T; it is
// described without arrays (cu_n == nullptr) and the helpers reduce to those closed forms.
// Masked layout (edm_s2a_bind_masked, speech editing): the P_s prompt ("known") rows of a sequence may sit anywhere among its N_s rows,
// not only in front. Two more arrays say where: tgt_enc maps target row -> encoder row, enc_slot maps encoder row -> target index t
// (>= 0) or -1 - k for the sequence's k-th known row in time order; per-sequence prompt data (tokens, codes, projected injections) keeps
// the known rows in that order. Without these arrays (every other bind) the known rows are the prefix and the helpers keep their
// closed forms.
#pragma once

namespace edm {

struct SeqLayout {
  int n_seq;
  int N, T;          // uniform layout: rows / target rows of every sequence (unused when cu_n != nullptr)
  const int* cu_n;   // [n_seq + 1] first encoder row of each sequence, cu_n[n_seq] = total rows; nullptr: uniform
  const int* cu_t;   // [n_seq + 1] first target row of each sequence
  int rows, t_rows;  // totals (sum N_s, sum T_s), for the host side of a launch
  const int* tgt_enc = nullptr;   // [t_rows] encoder row of every target row; nullptr: target t of sequence s is row n_start(s) + p_len(s) + t
  const int* enc_slot = nullptr;  // [rows] target index, or -1 - (index among the sequence's known rows); nullptr: the known rows are the prefix

  __device__ __forceinline__ bool packed() const { return cu_n != nullptr; }
  __device__ __forceinline__ int n_start(int s) const { return packed() ? __ldg(cu_n + s) : s * N; }
  __device__ __forceinline__ int n_len(int s) const { return packed() ? __ldg(cu_n + s + 1) - __ldg(cu_n + s) : N; }
  __device__ __forceinline__ int t_start(int s) const { return packed() ? __ldg(cu_t + s) : s * T; }
  __device__ __forceinline__ int t_len(int s) const { return packed() ? __ldg(cu_t + s + 1) - __ldg(cu_t + s) : T; }
  __device__ __forceinline__ int p_start(int s) const { return n_start(s) - t_start(s); }
  __device__ __forceinline__ int p_len(int s) const { return n_len(s) - t_len(s); }

  // last s with cu[s] <= i (n_seq <= a few hundred: a binary search over L1-resident offsets)
  __device__ __forceinline__ int search(const int* cu, int i) const {
    int lo = 0, hi = n_seq - 1;
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (__ldg(cu + mid) <= i) lo = mid; else hi = mid - 1;
    }
    return lo;
  }
  // encoder row -> (sequence, position inside it)
  __device__ __forceinline__ void enc_pos(int row, int& s, int& n) const {
    if (packed()) {
      s = search(cu_n, row);
      n = row - __ldg(cu_n + s);
    } else {
      s = row / N;
      n = row - s * N;
    }
  }
  // target row -> (sequence, target index t); its encoder row is enc_row(s, t)
  __device__ __forceinline__ void tgt_pos(int r, int& s, int& t) const {
    if (packed()) {
      s = search(cu_t, r);
      t = r - __ldg(cu_t + s);
    } else {
      s = r / T;
      t = r - s * T;
    }
  }
  __device__ __forceinline__ long long enc_row(int s, int t) const {
    if (tgt_enc != nullptr) return __ldg(tgt_enc + t_start(s) + t);
    return static_cast<long long>(n_start(s)) + p_len(s) + t;
  }
  // encoder row `row` (position n of sequence s, from enc_pos) -> its target index t >= 0, or -1 - k when it is the sequence's k-th
  // known row (prompt data of sequence s at p_start(s) + k)
  __device__ __forceinline__ int slot(int row, int s, int n) const {
    if (enc_slot != nullptr) return __ldg(enc_slot + row);
    const int np = p_len(s);
    return n < np ? -1 - n : n - np;
  }
  // element (q, t) of sequence s in a buffer of per-sequence [Q, T_s] blocks
  __device__ __forceinline__ long long out_offset(int s, int q, int Q, int t) const {
    return static_cast<long long>(Q) * t_start(s) + static_cast<long long>(q) * t_len(s) + t;
  }
  // Philox counter of target row t of sequence s when the batch starts at global sequence index seq0: (seq0 + s) T_s + t, what a
  // single-utterance call for sequence seq0 + s draws
  __device__ __forceinline__ long long philox_row(long long seq0, int s, int t) const { return (seq0 + s) * t_len(s) + t; }
};

inline SeqLayout uniform_layout(int n_seq, int N, int T) {
  SeqLayout l;
  l.n_seq = n_seq; l.N = N; l.T = T; l.cu_n = nullptr; l.cu_t = nullptr; l.rows = n_seq * N; l.t_rows = n_seq * T;
  return l;
}

}  // namespace edm
