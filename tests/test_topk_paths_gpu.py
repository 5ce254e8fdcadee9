"""Every branch of the TopK selection and of the k-sparse decode against the fp64 oracle (oracle/sae_oracle.py), run in
fp64 on the GPU.

Which branch a row takes is decided per plan and per row; the cases below reach each of them on purpose:

  branch (kernel condition)                                                          reached by
  selection from the chunk maxima of the scores epilogue: `fused` in                 1 (SCE_TOPK_CMAX=1), 2, 3 (duplicated
    topk_select2_kernel = chunk maxima written, k <= 256, j_pick = ceil(k /            halves at n = 2048, k = 7 / 33), 6
    full_warps) <= 32 with full_warps = min(8, n_chunks / 32)                         (n = 1048: 33 chunks, the last one
                                                                                      partial, one full warp)
  selection reading the row twice: not `fused` (n < 1024, k too large for the        1 (SCE_TOPK_CMAX=0), 1 (k = 64 at
    full warps, SCE_TOPK_CMAX=0)                                                      n = 4096), 5, 6 (n = 512)
  rank counting with parts == 1: ncand == kTopkCand (1024)                           3 (identical rows, n = 1024), 4 (k > 256
                                                                                      at n = 1024: every key is a candidate)
  4-pass radix select + ordered compaction: ncand > kTopkCand                        3 (identical rows at n = 2048, 1500
                                                                                      tied copies; all-zero / all-negative
                                                                                      rows), 4 (k > 256 at n = 3072)
  no k-sparse lists, every row zeroed in full: topk_k_max > 256 (topk_kmax() = 0)    2 (k = 257), 4
  k-sparse gather decode / code gradient (topk_sparse_kernel,                        1, 2, 5, 6, 7, 8, 9, 10
    topk_dz_scatter_kernel): SCE_TOPK_SPARSE or n >= 96 k_max, topk_slices > 0
  2 / 4 / 8 slices of the width (topk_slices, SCE_TOPK_SLICES)                       1 (4, 8 forced), 6 (d = 24: 2 slices
                                                                                      of 3 float4 groups; d = 4096: 8 only)
  no slice fits, dense decode although forced                                       6 (d = 4096 with k_max = 48; d = 5120)
  k classes {16, 32, 64, k_max} of the gather launches, list capacity rounded to 8   2, 9 (k lowered 64 -> 16)
  dense decode with lists kept: lists, n < 96 k_max or SCE_TOPK_SPARSE=0             1, 5, 7, 8
  per-model batches (x_model_stride of the gather kernel)                            8
  stale list entries on one plan across calls with different B                      7
  lowest-index tie-break on the chunk-maxima and on the radix path                   3
  refresh(): re-derived fp32 dictionary copy; k_max raised / lowered -> new plan     9
  k < 1, k > n rejected before any kernel runs                                       11

Every call is checked by `check_call`: the support must be a valid top-k of the fp64 scores (at most k positives per
row, lowest kept >= highest dropped clamped at 0, up to 1e-4 max|S|), hold min(k, positive fp64 scores) entries outside
a rounding window, and on that support x̂ and the code agree to 1e-4 norm-relative, the loss to 1e-4 and the dictionary
gradient to 2e-4 norm-relative (the bars of tests/test_engine_gpu.py).
"""
import pytest
import torch

from oracle import sae_oracle as O

pytestmark = pytest.mark.gpu

REL = 1e-4
GRAD_REL = 2e-4
ARITHS = ["f16f8", "bf16x3"]
KNOBS = ("SCE_TOPK_SPARSE", "SCE_TOPK_CMAX", "SCE_TOPK_SLICES")


def relnorm(a, b):
    a, b = a.double(), b.double().to(a.device)
    return float((a - b).norm() / b.norm().clamp(min=1e-30))


def relabs(a, b):
    return abs(float(a) - float(b)) / max(abs(float(b)), 1e-30)


def set_path(monkeypatch, sparse=None, cmax=None, slices=None):
    """Plan-time knobs of the selection / decode path; read when the plan is built, i.e. on the ensemble's first call."""
    for name, v in zip(KNOBS, (sparse, cmax, slices)):
        if v is None:
            monkeypatch.delenv(name, raising=False)
        else:
            monkeypatch.setenv(name, str(v))


def topk_models(dicts, ks):
    return [({"dict": D.float().contiguous().clone()}, {"sparsity": torch.tensor(int(k), dtype=torch.long)})
            for D, k in zip(dicts, ks)]


def random_models(d, n, ks, seed):
    gen = torch.Generator().manual_seed(seed)
    return topk_models([torch.randn(n, d, generator=gen) for _ in ks], ks)


def ensemble(models, arith):
    import sparse_coding_b200 as S
    clone = [({k: v.clone() for k, v in p.items()}, {k: v.clone() for k, v in b.items()}) for p, b in models]
    return S.FunctionalEnsemble(clone, S.TopKEncoder, S.adam, {"lr": 1e-3}, device="cuda", no_stacking=True, arith=arith)


def batch(B, d, seed, M=None):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    shape = (B, d) if M is None else (M, B, d)
    return torch.randn(*shape, generator=gen, device="cuda")


def check_call(tag, ens, X, code, loss, x_hat=None, grads=None, params=None, expand_dims=True):
    """One engine call (its code, loss and, if given, x̂ and gradients) against the fp64 oracle on `params` (default:
    the ensemble's current parameters). Returns the fp64 scores of every model."""
    params = ens.params["dict"] if params is None else params
    Xd = X.double()
    inf = float("inf")
    scores = []
    for m in range(ens.n_models):
        k = int(ens.buffers["sparsity"][m])
        Xm = Xd if expand_dims else Xd[m]
        support = code[m] > 0
        f = O.topk_grads(params[m].double(), Xm, k, support=support)
        S = f["Z"]
        tol = 1e-4 * float(S.abs().max())
        npos = support.sum(-1)
        assert int(npos.max()) <= k, (tag, m, int(npos.max()), k)
        kept = torch.where(support, S, torch.full_like(S, inf)).min(-1).values
        dropped = torch.where(support, torch.full_like(S, -inf), S).max(-1).values
        assert bool((kept >= dropped.clamp(min=0) - tol).all()), (tag, m, float((dropped.clamp(min=0) - kept).max()))
        lo, hi = (S > tol).sum(-1).clamp(max=k), (S > -tol).sum(-1).clamp(max=k)
        assert bool(((npos >= lo) & (npos <= hi)).all()), (tag, m, "positives per row != min(k, positive scores)")
        e = {"code": relnorm(code[m], f["c"]), "loss": relabs(loss["loss"][m], f["loss"])}
        if x_hat is not None:
            e["x_hat"] = relnorm(x_hat[m], f["x_hat"])
        if grads is not None:
            e["grad"] = relnorm(grads["dict"][m], f["grads"]["dict"])
        print(f"{tag} m={m} k={k} " + " ".join(f"{name} {v:.2e}" for name, v in e.items()))
        assert all(v <= REL for name, v in e.items() if name != "grad"), (tag, m, e)
        assert e.get("grad", 0.0) <= GRAD_REL, (tag, m, e)
        scores.append(S)
        del f
    return scores


def run_checked(tag, ens, X, expand_dims=True):
    """grads_batch + forward_batch(return_x_hat=True) on X, both checked; returns (dense code, fp64 scores, grads)."""
    grads, (loss, aux) = ens.grads_batch(X, expand_dims)
    code = aux["c"].dense()
    nnz = aux["c"].count_nonzero(dim=-1).float().mean(dim=-1)
    assert torch.allclose(nnz, code.count_nonzero(dim=-1).float().mean(dim=-1), rtol=1e-6), tag
    loss_f, aux_f, x_hat = ens.forward_batch(X, expand_dims, return_x_hat=True)
    assert torch.equal(aux_f["c"].dense(), code), tag
    assert torch.allclose(loss_f["loss"], loss["loss"], rtol=1e-6), tag
    scores = check_call(tag, ens, X, code, loss, x_hat=x_hat, grads=grads, expand_dims=expand_dims)
    return code, scores, grads


# ---------------------------------------------------------------------------------------------------------------------
# 1. path equivalence
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("arith", ARITHS)
def test_paths_agree_bitwise(arith, monkeypatch):
    """Selection does not depend on the decode path or on where the bound came from: every setting must give the
    bitwise same dense code, and each is checked against the oracle (k = 1 .. 64 at n = 4096: k = 64 is past the
    chunk-maxima path's 32 per full warp, so that model reads its rows twice even with SCE_TOPK_CMAX=1)."""
    d, n, B = 256, 4096, 300
    models = random_models(d, n, (1, 16, 33, 64), seed=10)
    X = batch(B, d, seed=11)
    settings = [dict(sparse=s, cmax=c) for s in (0, 1) for c in (0, 1)] + [dict(sparse=1, cmax=1, slices=sl) for sl in (4, 8)]
    first = None
    for st in settings:
        set_path(monkeypatch, **st)
        ens = ensemble(models, arith)
        code, _, _ = run_checked(f"paths {arith} {st}", ens, X)
        if first is None:
            first = code
        else:
            assert torch.equal(code, first), (st, int((code != first).sum()))
        del ens


# ---------------------------------------------------------------------------------------------------------------------
# 2. k classes and list capacity
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("arith", ARITHS)
def test_k_classes_and_list_capacity(arith, monkeypatch):
    """Every class boundary of the gather launches (16 | 17, 32 | 33, 64 | 65, the k_max class), both sides of the
    capacity round-up to 8 (7, 17, 33, 65, 120), and k = 256 (largest with lists) against k = 257 (no lists, rows
    zeroed in full) on the same data; then the gather path as the unforced heuristic picks it (n >= 96 k_max)."""
    d, n, B = 128, 8192, 64
    ks = (1, 7, 16, 17, 32, 33, 64, 65, 120, 256)
    set_path(monkeypatch, sparse=1)
    run_checked(f"classes {arith}", ensemble(random_models(d, n, ks, seed=20), arith), batch(B, d, seed=21))
    gen = torch.Generator().manual_seed(22)
    D = torch.randn(n, d, generator=gen)
    X = batch(B, d, seed=23)
    codes = {}
    for k in (256, 257):
        ens = ensemble(topk_models([D], [k]), arith)
        codes[k], _, _ = run_checked(f"k={k} {arith}", ens, X)
        run_checked(f"k={k} {arith} second batch", ens, batch(B // 2, d, seed=24))
    # the 257 code is the 256 code plus each row's 257th largest score (when positive)
    extra = (codes[257] != 0) & (codes[256] == 0)
    assert torch.equal(torch.where(extra, torch.zeros_like(codes[257]), codes[257]), codes[256])
    assert int(extra.sum(-1).max()) <= 1
    set_path(monkeypatch)
    ens = ensemble(random_models(d, n, (8, 40, 80), seed=25), arith)     # 96 * 80 <= 8192: gather path by default
    run_checked(f"heuristic {arith}", ens, X)


# ---------------------------------------------------------------------------------------------------------------------
# 3. radix fallback and ties, with the exact result known
# ---------------------------------------------------------------------------------------------------------------------
def _tie_batch(v, B, seed):
    """Rows a v + noise (a in [0.5, 2), so that x . v > 0), with every 8th row (from 3) all-zero and every 8th (from 5)
    negated; against a dictionary of copies of v all scores of a row tie. Returns (X, rows with positive scores).
    (The noise keeps the dictionary gradient away from zero: with x parallel to v it is exactly zero, all of dW lying
    along the normalised row, which the row-norm Jacobian projects out.)"""
    gen = torch.Generator(device="cuda").manual_seed(seed)
    a = 0.5 + 1.5 * torch.rand(B, 1, generator=gen, device="cuda")
    X = a * v.cuda()[None, :] + 0.5 * torch.randn(B, v.numel(), generator=gen, device="cuda")
    r = torch.arange(B, device="cuda")
    X[r % 8 == 3] = 0.0
    X[r % 8 == 5] *= -1.0
    return X, (r % 8 != 3) & (r % 8 != 5)


@pytest.mark.parametrize("arith", ARITHS)
@pytest.mark.parametrize("n", [2048, 1024])
def test_all_scores_tied_keep_lowest_columns(arith, n, monkeypatch):
    """A dictionary of n identical rows: every score of a row ties. n = 2048 puts 2048 keys at the bound (radix select),
    n = 1024 exactly kTopkCand (rank counting with parts == 1). The code must be the score on columns 0..k-1 and zero
    elsewhere; all-zero and all-negative rows must give a zero code, a zero x̂ and no gradient."""
    d, B = 128, 64
    set_path(monkeypatch, sparse=1)
    v = torch.randn(d, generator=torch.Generator().manual_seed(30))
    ks = (5, 100, 256)
    ens = ensemble(topk_models([v.repeat(n, 1)] * len(ks), ks), arith)
    X, pos = _tie_batch(v, B, seed=31)
    code, scores, _ = run_checked(f"ties n={n} {arith}", ens, X)
    for m, k in enumerate(ks):
        S = scores[m]
        want = torch.zeros_like(code[m])
        want[:, :k] = S[:, :k].float()
        want[~pos] = 0.0
        assert torch.equal(code[m] != 0, want != 0), (n, k, "columns other than 0..k-1 selected")
        assert relnorm(code[m], want) <= REL and float(((code[m] - want).abs() / S.abs().clamp(min=1e-30)).max()) <= REL
    # rows with nothing positive: exactly nothing out
    Xz = X[~pos].contiguous()
    grads, (loss, aux) = ens.grads_batch(Xz)
    assert int(aux["c"].dense().count_nonzero()) == 0
    assert int(grads["dict"].count_nonzero()) == 0
    _, _, x_hat = ens.forward_batch(Xz, return_x_hat=True)
    assert int(x_hat.count_nonzero()) == 0


@pytest.mark.parametrize("arith", ARITHS)
def test_tie_block_among_random_rows(arith, monkeypatch):
    """1500 copies of one row interleaved among 548 random rows (n = 2048): inputs along that row rank the copies
    first, so k cuts through a 1500-way tie (radix select) and must keep the lowest-index copies."""
    d, n, B = 128, 2048, 64
    set_path(monkeypatch, sparse=1)
    gen = torch.Generator().manual_seed(40)
    u = torch.randn(d, generator=gen)
    tie = torch.randperm(n, generator=gen)[:1500].sort().values
    D = torch.randn(n, d, generator=gen)
    D[tie] = u
    ks = (37, 256)
    ens = ensemble(topk_models([D] * len(ks), ks), arith)
    g = torch.Generator(device="cuda").manual_seed(41)
    X = (0.5 + 1.5 * torch.rand(B, 1, generator=g, device="cuda")) * u.cuda() + 0.3 * torch.randn(B, d, generator=g, device="cuda")
    X[::7] = 0.0
    code, scores, _ = run_checked(f"tie block {arith}", ens, X)
    tie_c = tie.cuda()
    other = torch.ones(n, dtype=torch.bool, device="cuda")
    other[tie_c] = False
    for m, k in enumerate(ks):
        S = scores[m]
        t = S[:, tie_c[0]]
        above = (S[:, other] > t[:, None]).sum(-1)
        for r in range(B):
            if r % 7 == 0:
                assert int(code[m, r].count_nonzero()) == 0
                continue
            assert int(above[r]) < k and float(t[r]) > 0
            want = torch.zeros(n, dtype=torch.bool, device="cuda")
            want[other.nonzero().flatten()[S[r, other] > t[r]]] = True
            want[tie_c[: k - int(above[r])]] = True
            assert torch.equal(code[m, r] > 0, want), (k, r)


@pytest.mark.parametrize("arith", ARITHS)
def test_duplicated_halves_on_chunk_maxima_path(arith, monkeypatch):
    """test_engine_gpu's duplicated-halves tie test at n = 2048 (64 chunks, two full warps of chunk maxima: k = 7 and
    33 are both selected from the chunk maxima): row j == row j + 1024, so an odd k cuts through a pair, and of a
    tied pair the lower column must be kept."""
    d, n, B = 128, 2048, 96
    set_path(monkeypatch, sparse=1, cmax=1)
    half = torch.randn(n // 2, d, generator=torch.Generator().manual_seed(50))
    ks = (7, 33)
    ens = ensemble(topk_models([torch.cat([half, half])] * 2, ks), arith)
    code, scores, _ = run_checked(f"dup halves {arith}", ens, batch(B, d, seed=51))
    for m, k in enumerate(ks):
        sel = code[m] > 0
        assert bool((sel.sum(-1) == k).all())          # (randn rows: far more than k positive scores)
        lo, hi = sel[:, : n // 2], sel[:, n // 2:]
        assert bool((~hi | lo).all()), (k, "an upper copy kept without its lower twin")
        assert bool((lo.sum(-1) == (k + 1) // 2).all()) and bool((hi.sum(-1) == k // 2).all())


# ---------------------------------------------------------------------------------------------------------------------
# 4. k > 256 and k = n
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("arith", ARITHS)
@pytest.mark.parametrize("n", [1024, 3072])
def test_k_above_list_capacity(arith, n, monkeypatch):
    """k > 256: no lists, every key a candidate (n = 1024: exactly kTopkCand, rank counting; n = 3072: radix select).
    At k = n the code is relu(scores)."""
    d, B = 128, 64
    set_path(monkeypatch)
    ks = (257, 512, n) if n == 1024 else (257, 512)
    ens = ensemble(random_models(d, n, ks, seed=60 + n), arith)
    code, scores, _ = run_checked(f"k>256 n={n} {arith}", ens, batch(B, d, seed=61))
    run_checked(f"k>256 n={n} {arith} second batch", ens, batch(B // 2 + 1, d, seed=62))
    if n == 1024:
        assert relnorm(code[2], scores[2].clamp(min=0)) <= REL


# ---------------------------------------------------------------------------------------------------------------------
# 5. fewer than k positive scores
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("arith", ARITHS)
@pytest.mark.parametrize("sparse", [0, 1])
@pytest.mark.parametrize("d,n,k", [(64, 64, 48), (128, 512, 256)])
def test_fewer_positive_scores_than_k(arith, sparse, d, n, k, monkeypatch):
    """Inputs against the dictionary's common direction: most scores are negative, so the selection keeps negative
    scores, which must add nothing to x̂, the loss or the gradient (the gather kernel and the code-gradient scatter
    skip them)."""
    B = 64
    set_path(monkeypatch, sparse=sparse)
    gen = torch.Generator().manual_seed(70 + n)
    e = torch.randn(d, generator=gen)
    e /= e.norm()
    D = torch.randn(n, d, generator=gen) + 4.0 * e
    ens = ensemble(topk_models([D], [k]), arith)
    X = batch(B, d, seed=71) - 4.0 * e.cuda()
    code, scores, _ = run_checked(f"few positives n={n} k={k} sparse={sparse} {arith}", ens, X)
    assert int((scores[0] > 0).sum(-1).max()) < k     # the case is what it claims to be


# ---------------------------------------------------------------------------------------------------------------------
# 6. widths
# ---------------------------------------------------------------------------------------------------------------------
WIDTHS = [
    # (d, n, ks, ariths)
    (8, 512, (4, 16), ["bf16x3"]),            # one float4 group per slice
    (24, 512, (4, 16), ["bf16x3"]),           # 2 slices of 3 float4 groups
    (4096, 1024, (8, 40), ARITHS),            # 8 slices of 512 columns: fits up to k_max = 40
    (4096, 1024, (8, 48), ARITHS),            # k_max = 48 does not fit: dense decode although forced
    (5120, 1024, (8, 16), ARITHS),            # no slice count fits: dense decode
    (128, 1048, (8, 32, 33), ["bf16x3"]),     # 33 chunks of 32 columns, the last one partial (one full warp)
]


@pytest.mark.parametrize("case", [(w, a) for w in WIDTHS for a in w[3]], ids=lambda c: f"d{c[0][0]}-n{c[0][1]}-k{max(c[0][2])}-{c[1]}")
def test_widths_with_sparse_forced(case, monkeypatch):
    (d, n, ks, _), arith = case
    set_path(monkeypatch, sparse=1)
    ens = ensemble(random_models(d, n, ks, seed=80 + d), arith)
    run_checked(f"width d={d} n={n} {arith}", ens, batch(64, d, seed=81))
    ens.step_batch(batch(64, d, seed=82))
    run_checked(f"width d={d} n={n} {arith} after a step", ens, batch(40, d, seed=83))


# ---------------------------------------------------------------------------------------------------------------------
# 7. state across calls on one plan
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("arith", ARITHS)
@pytest.mark.parametrize("sparse", [0, 1])
def test_state_across_calls_with_changing_batch(arith, sparse, monkeypatch):
    """One plan, calls with B = 300, 37, 300, 129, 1, ... interleaving forward, gradients and steps: the lists of the
    previous call (possibly of a larger B) must be cleared exactly, every call checked on the parameters it saw."""
    d, n = 128, 2048
    set_path(monkeypatch, sparse=sparse)
    ens = ensemble(random_models(d, n, (8, 24, 64), seed=90), arith)
    seq = [(300, "grads"), (37, "step"), (300, "forward"), (129, "step"), (1, "grads"), (300, "step"), (37, "forward"),
           (1, "step")]
    for i, (B, kind) in enumerate(seq):
        X = batch(B, d, seed=91 + i)
        tag = f"state {arith} sparse={sparse} call {i} B={B} {kind}"
        if kind == "grads":
            grads, (loss, aux) = ens.grads_batch(X)
            code = aux["c"].dense()
            check_call(tag, ens, X, code, loss, grads=grads)
        elif kind == "forward":
            loss, aux, x_hat = ens.forward_batch(X, return_x_hat=True)
            code = aux["c"].dense()
            check_call(tag, ens, X, code, loss, x_hat=x_hat)
        else:
            before = ens.params["dict"].clone()
            loss, aux = ens.step_batch(X)
            code = aux["c"].dense()
            check_call(tag, ens, X, code, loss, params=before)
        counts = ens.active_counts(B)
        assert torch.equal(counts, (code != 0).sum(1, dtype=torch.int32)), tag


# ---------------------------------------------------------------------------------------------------------------------
# 8. per-model batches
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("arith", ARITHS)
@pytest.mark.parametrize("sparse", [0, 1])
def test_per_model_batches(arith, sparse, monkeypatch):
    d, n, B = 128, 4096, 96
    set_path(monkeypatch, sparse=sparse)
    ens = ensemble(random_models(d, n, (8, 33, 64), seed=100), arith)
    run_checked(f"per-model {arith} sparse={sparse}", ens, batch(B, d, seed=101, M=3), expand_dims=False)
    ens.step_batch(batch(B, d, seed=102, M=3), expand_dims=False)
    run_checked(f"per-model {arith} sparse={sparse} after a step", ens, batch(B - 17, d, seed=103, M=3), expand_dims=False)


# ---------------------------------------------------------------------------------------------------------------------
# 9. refresh()
# ---------------------------------------------------------------------------------------------------------------------
def _three_calls(tag, ens, d, seed):
    """grads, forward and a step on fresh batches, each checked (at most k non-zeros per row: check_call)."""
    run_checked(f"{tag} call 1", ens, batch(200, d, seed=seed))
    X = batch(77, d, seed=seed + 1)
    before = ens.params["dict"].clone()
    loss, aux = ens.step_batch(X)
    check_call(f"{tag} call 2 (step)", ens, X, aux["c"].dense(), loss, params=before)
    run_checked(f"{tag} call 3", ens, batch(150, d, seed=seed + 2))


@pytest.mark.parametrize("arith", ARITHS)
def test_refresh_rederives_edited_dictionary(arith, monkeypatch):
    """Dictionary rows edited from outside: refresh() must re-derive the gather path's fp32 normalised copy."""
    d, n = 128, 4096
    set_path(monkeypatch, sparse=1)
    ens = ensemble(random_models(d, n, (8, 32), seed=110), arith)
    run_checked(f"refresh edit {arith} before", ens, batch(200, d, seed=111))
    gen = torch.Generator(device="cuda").manual_seed(112)
    with torch.no_grad():
        ens.params["dict"][:, : n // 2] = 3.0 * torch.randn(2, n // 2, d, generator=gen, device="cuda")
    ens.refresh()
    _three_calls(f"refresh edit {arith}", ens, d, seed=113)


@pytest.mark.parametrize("arith", ARITHS)
def test_refresh_after_raising_k_past_capacity(arith, monkeypatch):
    """k = (8, 16) planned (list capacity 16), then model 0 raised to k = 40 and refresh(): the plan must follow the new
    k_max, else the selection scatters 40 entries and records 16, the decode reads 16 and the other 24 stay behind."""
    d, n = 128, 4096
    set_path(monkeypatch, sparse=1)
    ens = ensemble(random_models(d, n, (8, 16), seed=120), arith)
    run_checked(f"raise k {arith} before", ens, batch(200, d, seed=121))
    ens.buffers["sparsity"][0] = 40
    ens.refresh()
    _three_calls(f"raise k {arith}", ens, d, seed=122)


@pytest.mark.parametrize("arith", ARITHS)
def test_refresh_after_lowering_k(arith, monkeypatch):
    """k lowered across a class boundary (64 -> 16): first with k_max unchanged (the classes are regrouped on the same
    plan), then with k_max lowered (a new plan)."""
    d, n = 128, 4096
    set_path(monkeypatch, sparse=1)
    ens = ensemble(random_models(d, n, (64, 64, 32), seed=130), arith)
    run_checked(f"lower k {arith} before", ens, batch(200, d, seed=131))
    ens.buffers["sparsity"][0] = 16
    ens.refresh()
    _three_calls(f"lower k {arith} same k_max", ens, d, seed=132)
    ens.buffers["sparsity"][1] = 16
    ens.refresh()
    _three_calls(f"lower k {arith} k_max 32", ens, d, seed=136)


# ---------------------------------------------------------------------------------------------------------------------
# 10. trajectory on the gather path
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("arith", ARITHS)
def test_gather_path_trajectory(arith, monkeypatch):
    """20 Adam steps on the gather path against the reference step (fp32, per-model loop) on the same GPU."""
    d, n, B = 128, 4096, 256
    set_path(monkeypatch, sparse=1)
    models = random_models(d, n, (8, 32, 96), seed=140)
    ens = ensemble(models, arith)
    cuda = [({k: v.cuda() for k, v in p.items()}, {k: v.cuda() for k, v in b.items()}) for p, b in models]
    ref = O.RefPortEnsemble(cuda, O.SIG_LOSSES["topk"], lr=1e-3, no_stacking=True)
    for step in range(20):
        X = batch(B, d, seed=141 + step)
        loss, _ = ens.step_batch(X)
        rloss, _ = ref.step_batch(X)
        assert torch.allclose(loss["loss"], rloss["loss"], rtol=1e-3), (step, loss["loss"], rloss["loss"])
    e = relnorm(ens.params["dict"], ref.params["dict"])
    print(f"trajectory {arith}: |dict - ref| / |ref| = {e:.2e}")
    assert e <= 2e-3


# ---------------------------------------------------------------------------------------------------------------------
# 11. validation
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("bad", [0, -3, 513])
def test_k_outside_range_is_rejected(bad, monkeypatch):
    """k < 1 or k > n raises ValueError naming the model, on the first call and on refresh(), before any kernel runs;
    the library itself refuses a k above the plan's topk_k_max."""
    import ctypes as C

    from sparse_coding_b200 import _lib
    d, n = 64, 512
    set_path(monkeypatch)
    ens = ensemble(random_models(d, n, (8, 16), seed=150), "auto")
    ens.buffers["sparsity"][1] = bad
    with pytest.raises(ValueError, match="model 1"):
        ens.forward_batch(batch(32, d, seed=151))
    ens.buffers["sparsity"][1] = 16
    run_checked("validation", ens, batch(32, d, seed=152))
    ens.buffers["sparsity"][1] = bad
    with pytest.raises(ValueError, match="model 1"):
        ens.refresh()
    ens.buffers["sparsity"][1] = 16
    ens.refresh()
    run_checked("validation after refresh", ens, batch(32, d, seed=153))
    # the engine's own check: its copy of the sparsity buffer holds a k above topk_k_max = 16
    ens._engine_buffers["sparsity"][0] = 17
    lib = _lib.load()
    rc = lib.sce_prepare(ens._plan, C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc != 0 and b"model 0" in lib.sce_last_error()
    ens._engine_buffers["sparsity"][0] = 8
    assert lib.sce_prepare(ens._plan, C.c_void_p(torch.cuda.current_stream().cuda_stream)) == 0
    run_checked("validation after the engine's refusal", ens, batch(32, d, seed=154))
