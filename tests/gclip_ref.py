"""Reference of Knet's per-tensor gradient clipping, update!(w, g, ::Adam) -> gclip!(g, gclip), on top of the oracle's Adam
(oracle.update): tensor k's gradient is scaled by (float32)(gclip / |g_k|) when |g_k| > gclip, |g_k| accumulated in fp64."""
import numpy as np

from oracle import lrcn_oracle as O


def norms(gloss):
    return np.array([np.sqrt(np.sum(np.square(g, dtype=np.float64))) for g in gloss])


def clip(gloss, gclip):
    """The gradients Adam sees: new arrays for the clipped tensors, the caller's arrays are never modified."""
    out = []
    for g, n in zip(gloss, norms(gloss)):
        out.append(g * np.float32(gclip / n) if gclip > 0 and n > gclip else g)
    return out


def update(param, gloss, optim, gclip=0.0):
    O.update(param, clip(gloss, gclip), optim)


def pick_gclip(nrm, avoid=None):
    """A threshold in the widest gap between sorted norms that leaves at least three tensors on each side (geometric middle of
    the gap); `avoid`: a threshold already used, whose gap is skipped."""
    s = np.sort(np.asarray(nrm, np.float64))
    best = None
    for i in (2, 3, 4, 5):
        t = float(np.sqrt(s[i] * s[i + 1]))
        if avoid is not None and s[i] < avoid < s[i + 1]:
            continue
        if best is None or s[i + 1] / s[i] > best[0]:
            best = (s[i + 1] / s[i], t)
    return best[1]
