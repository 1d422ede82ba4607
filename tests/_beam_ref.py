"""Plain-Python (numpy, float64) restatement of the CTC prefix beam search of k_ctc_beam_decode (csrc/ctc.cu), the yardstick
of the beam decoder (tests only).

Per frame the input is log(p + 1e-7) followed by a log-softmax over the C classes [TF-SEMANTICS: K.ctc_decode(greedy=False)
feeds log(y_pred + 1e-7) to tf.nn.ctc_beam_search_decoder, which treats it as logits].  Blank = C - 1.  A beam is a prefix
with (log P_blank, log P_label), its total, its parent (the kept beam one symbol shorter, or -1) and its last symbol.  At
frame t every kept beam b of rank r gives its continuation (candidate index r C + C - 1) and its extensions by c < C - 1
(index r C + c) whose prefix is not already a kept beam (a kept beam with parent b and last symbol c); the beam_width
candidates with the largest total are kept, ties to the lower index, and candidates of total -inf are never kept."""
import numpy as np
import torch

KERAS_EPS = 1e-7


def _peaked_logits(seed, b, t, c):
    """Logits of a planted path (letters held over several frames, blanks, repeats) plus N(0, 1.5^2) noise: peaked
    probabilities with plausible competitors."""
    g = torch.Generator().manual_seed(seed)
    blank = c - 1
    path = torch.empty(b, t, dtype=torch.long)
    for i in range(b):
        prev = blank
        for s in range(t):
            u = float(torch.rand(1, generator=g))
            prev = prev if u < 0.45 else (blank if u < 0.7 else int(torch.randint(0, c, (1,), generator=g)))
            path[i, s] = prev
    z = torch.randn(b, t, c, generator=g) * 1.5
    z.scatter_add_(2, path.unsqueeze(-1), torch.full((b, t, 1), 5.0))
    return z


def frame_log_probs(p):
    """log-softmax(log(p + 1e-7)) over the last axis, float64."""
    lp = np.log(np.asarray(p, np.float64) + KERAS_EPS)
    m = lp.max(-1, keepdims=True)
    return lp - m - np.log(np.exp(lp - m).sum(-1, keepdims=True))


def _margin(flat, kept, pruned, c_num, last):
    """Smallest gap between a kept and a pruned candidate total (flat[kept], flat[pruned]) that may order differently in
    fp32.  An exact float64 tie at the boundary is resolved by the index rule the same way in any precision only when it is
    the same operation on equal operands: extensions of ONE beam by classes of equal probability, none of them the beam's
    last symbol (so each adds x[c] to the beam's total).  Then the margin is the gap to the nearest distinct totals; any other
    exact tie is a near-tie of margin 0."""
    kv, pv = flat[kept], flat[pruned]
    lo, hi = kv.min(), pv.max()
    if hi < lo:
        return lo - hi
    tied = np.concatenate([kept[kv == lo], pruned[pv == lo]])
    r, c = tied // c_num, tied % c_num
    if not (np.all(r == r[0]) and np.all(c != c_num - 1) and np.all(c != last[r[0]])):
        return 0.0
    above, below = kv[kv > lo], pv[pv < hi]
    return min(above.min() - lo if above.size else np.inf, hi - below.max() if below.size else np.inf)


def beam_decode_one(x, beam_width, top_paths=1, merge_repeated=True):
    """Beam search over x (T, C) per-frame log-probabilities.  Returns (paths, log_probs, margin): top_paths int lists (empty
    beyond the live beams), their totals (-inf beyond the live beams) and the smallest margin between the kept and the pruned
    candidates over all steps, and between consecutive beams of the first top_paths + 1 at the end (the output order)."""
    t_len, c_num = x.shape
    blank = c_num - 1
    pb, pl, tot = np.zeros(1), np.full(1, -np.inf), np.zeros(1)
    last, par = np.full(1, -1), np.full(1, -1)
    prefixes = [()]
    margin = np.inf
    for t in range(t_len):
        xt = x[t]
        nb = len(prefixes)
        # continuations
        npb = tot + xt[blank]
        npl = np.where(last >= 0, pl + xt[np.maximum(last, 0)], -np.inf)
        has_par = par >= 0
        pp = np.maximum(par, 0)
        prev = np.where(last == last[pp], pb[pp], tot[pp])
        npl = np.where(has_par, np.logaddexp(npl, prev + xt[np.maximum(last, 0)]), npl)
        ntot = np.logaddexp(npb, npl)
        # extensions; candidate index = position in the flattened (nb, C) table
        cand = xt[None, :] + np.where(np.arange(c_num)[None, :] == last[:, None], pb[:, None], tot[:, None])
        cand[par[has_par], last[has_par]] = -np.inf                                 # prefix already kept
        cand[:, blank] = ntot
        flat = cand.reshape(-1)
        valid = np.nonzero(flat > -np.inf)[0]
        order = valid[np.argsort(-flat[valid], kind="stable")]                      # ties -> lower index
        if order.size > beam_width:
            margin = min(margin, _margin(flat, order[:beam_width], order[beam_width:], c_num, last))
            order = order[:beam_width]
        r, c = order // c_num, order % c_num
        cont = c == blank
        contrank = np.full(nb, -1)
        contrank[r[cont]] = np.nonzero(cont)[0]
        new_par = np.where(cont, np.where(par[r] >= 0, contrank[np.maximum(par[r], 0)], -1), contrank[r])
        pb = np.where(cont, npb[r], -np.inf)
        pl = np.where(cont, npl[r], flat[order])
        tot = flat[order].copy()
        last = np.where(cont, last[r], c)
        par = new_par
        prefixes = [prefixes[ri] if ci == blank else prefixes[ri] + (int(ci),) for ri, ci in zip(r.tolist(), c.tolist())]
    for k in range(min(top_paths, len(prefixes) - 1)):   # output order; an exact tie here is taken as a near-tie
        margin = min(margin, tot[k] - tot[k + 1])
    paths, scores = [], []
    for k in range(top_paths):
        if k >= len(prefixes):
            paths.append([])
            scores.append(-np.inf)
            continue
        w = list(prefixes[k])
        if merge_repeated:                                   # [TF-SEMANTICS] tf v1 merges repeats of the decoded beam
            w = [a for i, a in enumerate(w) if i == 0 or w[i - 1] != a]
        paths.append(w)
        scores.append(float(tot[k]))
    return paths, np.array(scores), margin


def ctc_beam_decode(probs, input_length=None, beam_width=100, top_paths=1, merge_repeated=True):
    """K.ctc_decode(greedy=False) restated: probs (B, T, C) softmax probabilities, input_length (B,) frames (clamped to [0, T])
    or None.  Returns (paths, log_prob, margin): paths[k][b] int lists, log_prob (B, top_paths) float64, margin (B,)."""
    p = np.asarray(probs.detach().cpu() if isinstance(probs, torch.Tensor) else probs)
    b, t_max, _ = p.shape
    x = frame_log_probs(p)
    paths = [[None] * b for _ in range(top_paths)]
    log_prob, margin = np.zeros((b, top_paths)), np.zeros(b)
    for i in range(b):
        t_b = t_max if input_length is None else min(max(int(np.asarray(input_length).reshape(-1)[i]), 0), t_max)
        w, s, m = beam_decode_one(x[i, :t_b], beam_width, top_paths, merge_repeated)
        for k in range(top_paths):
            paths[k][i] = w[k]
        log_prob[i], margin[i] = s, m
    return paths, log_prob, margin


def labeling_log_probs(x):
    """Brute force over all C^T alignments of x (T, C) log-probabilities: {labeling tuple: log p(labeling | x)} with the
    CTC collapse (merge repeats, then drop blanks).  Only for tiny T and C."""
    t_len, c_num = x.shape
    acc = {}
    for path in np.ndindex(*([c_num] * t_len)):
        lab = tuple(a for i, a in enumerate(path) if a != c_num - 1 and (i == 0 or path[i - 1] != a))
        acc.setdefault(lab, []).append(sum(x[t, a] for t, a in enumerate(path)))
    return {k: float(np.logaddexp.reduce(v)) for k, v in acc.items()}
