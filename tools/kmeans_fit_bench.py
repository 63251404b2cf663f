"""K-means fit of the semantic tokenizer on one GPU (edm_tts_b200.kmeans.fit_kmeans, SemanticTokenizer.fit), with the card name and
power limit read in the same run. Data: a seeded mixture of 1024 Gaussian centres in 1024 dimensions plus noise, generated on the device.
  (a) 262 144 rows (faiss's default sample for k = 1024: 256 points per centroid), k = 1024, 25 iterations: ms per iteration, split
      into event-bracketed assign, update (sort + offsets + edm_kmeans_update + objective) and host (counts copy, splits, repack); the update
      kernel alone is timed again afterwards on the last assignment, with its algorithmic bytes / time against 7.7 TB/s of HBM;
  (b) the same on 2 097 152 rows (max_points_per_centroid=None);
  (c) the incumbent on the (a) rows and init: Lloyd's in plain torch (cdist + argmin + index_add_, fp32, TF32 off, chunked), its time
      and final objective next to ours;
  (d) SemanticTokenizer.fit on synthetic hubert-large weights, 64 clips of 3-20 s: feature extraction and fit timed separately.
(a) and (b) also record, on the final centroids, how far sum |x|^2 - 2 sum best from the assignment's fp32 scores lies from the exact
fp64 objective the fit records. Every case is warmed up once. Writes JSON to argv[1]. Fails without a GPU: there is nothing to fall back to."""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

K, D, NITER = 1024, 1024, 25
HBM_BYTES_PER_S = 7.7e12


def mixture(n, seed):
    """n rows: one of K Gaussian centres (unit variance per dimension) plus noise of std 0.5, on the device."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    centres = torch.randn(K, D, device="cuda", generator=g)
    x = torch.empty(n, D, device="cuda")
    for a in range(0, n, 1 << 18):
        b = min(n, a + (1 << 18))
        lab = torch.randint(0, K, (b - a,), device="cuda", generator=g)
        x[a:b] = centres[lab] + 0.5 * torch.randn(b - a, D, device="cuda", generator=g)
    return x


def update_bytes(n, k, dim):
    """Algorithmic HBM bytes of edm_kmeans_update: the rows once, perm + idx (8 B each per row), the fp64 partials written and read
    back, offsets, the centroids written."""
    slots = k + (n + 255) // 256
    return n * dim * 4 + 2 * n * 8 + 2 * slots * dim * 8 + (k + 1) * 8 + k * dim * 4


def fit_timed(x, init, niter=NITER):
    """One fit of NITER iterations through the Lloyd steps, assign and update bracketed with events: returns the state, the wall time
    of the iterations (ends in a synchronise) and the mean ms of assign / update per iteration; the rest of an iteration is host."""
    from edm_tts_b200.kmeans import prepare_fit

    run = prepare_fit(x, n_centroids=K, niter=niter, max_points_per_centroid=None, init=init)   # sum |x|^2 once: not per iteration
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ev = []
    for it in range(niter):
        e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        e[0].record()
        run.assign()
        e[1].record()
        run.update(it)
        e[2].record()
        run.split()          # the counts come to the host here: waits for assign + update
        run.repack()
        ev.append(e)
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) * 1e3
    assign = sum(e[0].elapsed_time(e[1]) for e in ev) / niter
    update = sum(e[1].elapsed_time(e[2]) for e in ev) / niter
    return run, wall, assign, update


def update_kernel_ms(run, reps=20):
    """edm_kmeans_update alone on the last assignment (sort and offsets outside the timed window)."""
    from edm_tts_b200 import _lib as L

    n, dim, k = run.n, run.dim, run.k
    srt, perm = torch.sort(run.idx, stable=True)
    offsets = torch.searchsorted(srt, torch.arange(k + 1, device="cuda", dtype=torch.int64))
    partials = torch.empty(L.lib().edm_kmeans_update_workspace_bytes(n, dim, k) // 8, device="cuda", dtype=torch.float64)
    c = run.centroids.clone()

    def call():
        L.check(L.lib().edm_kmeans_update(L.ptr(run.x), n, dim, L.ptr(run.idx), L.ptr(perm), L.ptr(offsets), k, L.ptr(partials), L.ptr(c),
                                          None, L.stream_ptr()), "kmeans_update")

    call()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        call()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def case_fit(name, x, init):
    fit_timed(x, init, niter=2)                                  # warm-up at the timed shapes: every kernel (sort included), the allocator
    run, wall, assign, update = fit_timed(x, init)
    n = x.shape[0]
    ms_k = update_kernel_ms(run)
    nb = update_bytes(n, K, D)
    # the objective the fit records (exact fp64 distances of the assignment) against sum |x|^2 - 2 sum best from the assignment's
    # fp32 scores, on the final centroids, relative to sum |x|^2
    idx, best = run.assigner.assign(run.x, return_scores=True)
    exact = sum((run.x[a:a + 65536].double() - run.centroids[idx[a:a + 65536]].double()).pow(2).sum() for a in range(0, n, 65536)).item()
    from_scores = (run.sq_total - 2.0 * best.double().sum()).item()
    r = dict(case=name, rows=n, k=K, dim=D, niter=NITER, ms_per_iter=round(wall / NITER, 3), assign_ms=round(assign, 3),
             update_ms=round(update, 3), host_ms=round(wall / NITER - assign - update, 3), update_share=round(update / (wall / NITER), 3),
             update_kernel_ms=round(ms_k, 3), update_kernel_bytes=nb, update_kernel_tb_s=round(nb / ms_k / 1e9, 2),
             update_kernel_frac_hbm=round(nb / ms_k / 1e9 / (HBM_BYTES_PER_S / 1e12), 3),
             objective_first=run.objective[0].item(), objective_last=run.objective[-1].item(), n_split=sum(run.n_split),
             final_objective_exact=exact, final_objective_from_scores=from_scores,
             from_scores_rel_err=abs(from_scores - exact) / run.sq_total.item())
    print(json.dumps(r), flush=True)
    return r, run


def torch_lloyd(x, init, chunk=32768):
    """The incumbent: Lloyd's in plain torch fp32 (TF32 off), cdist + argmin per chunk of rows, index_add_ means; empty clusters keep
    their centroid. Returns (centroids, objective per iteration before the update)."""
    c = init.clone()
    obj = []
    for _ in range(NITER):
        ids = torch.empty(x.shape[0], device="cuda", dtype=torch.int64)
        o = torch.zeros((), device="cuda", dtype=torch.float64)
        for a in range(0, x.shape[0], chunk):
            d = torch.cdist(x[a:a + chunk], c)
            m, i = d.min(1)
            ids[a:a + chunk] = i
            o += m.double().pow(2).sum()
        obj.append(o)
        s = torch.zeros_like(c).index_add_(0, ids, x)
        cnt = torch.zeros(c.shape[0], device="cuda").index_add_(0, ids, torch.ones(x.shape[0], device="cuda"))
        c = torch.where(cnt[:, None] > 0, s / cnt.clamp(min=1)[:, None], c)
    return c, [v.item() for v in obj]


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    if not torch.cuda.is_available():
        sys.exit("kmeans_fit_bench: no CUDA device; this benchmark runs on a B200 only (there is no CPU path to measure)")
    import __graft_entry__ as ge

    ge.build()
    from edm_tts_b200.kmeans import init_indices

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    rows = []
    # (a) and (c)
    xa = mixture(K * 256, 11)
    init = xa[init_indices(xa.shape[0], K, 1234).cuda()].clone()
    ra, run_a = case_fit("a_fit_262144x1024_k1024", xa, init)
    rows.append(ra)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch_lloyd(xa[:K * 4], init)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    _, obj_t = torch_lloyd(xa, init)
    torch.cuda.synchronize()
    ms_t = (time.perf_counter() - t0) * 1e3
    rc = dict(case="c_torch_lloyd_262144x1024_k1024", ms_per_iter=round(ms_t / NITER, 3), objective_last=obj_t[-1],
              ours_objective_last=ra["objective_last"], ours_ms_per_iter=ra["ms_per_iter"], speedup=round(ms_t / NITER / ra["ms_per_iter"], 2),
              objective_rel_diff=abs(obj_t[-1] - ra["objective_last"]) / obj_t[-1])
    print(json.dumps(rc), flush=True)
    rows.append(rc)
    del xa, run_a
    torch.cuda.empty_cache()
    # (b)
    xb = mixture(K * 2048, 12)
    init = xb[init_indices(xb.shape[0], K, 1234).cuda()].clone()
    rb, run_b = case_fit("b_fit_2097152x1024_k1024", xb, init)
    rows.append(rb)
    del xb, run_b
    torch.cuda.empty_cache()
    # (d)
    from edm_tts_b200 import HubertFeatures, SemanticTokenizer
    from edm_tts_b200.hubert import normalize_clip
    from edm_tts_b200.kmeans import fit_kmeans
    from edm_tts_b200.synthetic import hubert_config, make_hubert_state_dict

    cfg = hubert_config()
    hub = HubertFeatures(cfg, make_hubert_state_dict(0, cfg), device="cuda")
    g = torch.Generator().manual_seed(2024)
    lens = [int(v) for v in torch.randint(3 * 16000, 20 * 16000 + 1, (64,), generator=g)]
    clips = [torch.randn(n, generator=g).cuda() for n in lens]
    SemanticTokenizer.fit(hub, clips, n_centroids=K, niter=2)               # warm-up at the timed shapes

    def timed(fn):
        torch.cuda.synchronize()
        t = time.perf_counter()
        r = fn()
        torch.cuda.synchronize()
        return r, (time.perf_counter() - t) * 1e3

    feats, ms_feat = timed(lambda: torch.cat(hub.forward_batch([normalize_clip(c) for c in clips])))
    fit, ms_fit = timed(lambda: fit_kmeans(feats, n_centroids=K, niter=NITER, device="cuda"))
    (_, fit2), ms_all = timed(lambda: SemanticTokenizer.fit(hub, clips, n_centroids=K, niter=NITER))
    rd = dict(case="d_semantic_tokenizer_fit_64x3-20s", clips=64, frames=feats.shape[0], audio_s=round(sum(lens) / 16000, 1),
              features_ms=round(ms_feat, 2), fit_ms=round(ms_fit, 2), total_ms=round(ms_all, 2),
              same_centroids=bool(torch.equal(fit.centroids, fit2.centroids)), objective_last=fit.objective[-1], n_split=sum(fit.n_split))
    print(json.dumps(rd), flush=True)
    rows.append(rd)
    res = dict(card=smi, note="synthetic data and weights; CUDA events around assign / update, host clock (ending in a synchronise) "
                              "around whole fits; HBM figure 7.7 TB/s (data sheet)", cases=rows)
    if out_path:
        os.makedirs(os.path.dirname(out_path) or ".", exist_ok=True)
        with open(out_path, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
