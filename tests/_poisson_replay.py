"""numpy restatement of the engine's noise field (csrc/poisson.cuh) for exact comparisons.

The engine draws pixel `pixel` (= y * Nx + x) of image `image` (the orientation) from Philox4x32-10
counters (pixel lo, pixel hi, image, attempt) with key = seed: Knuth's multiplication method for
0 < lambda < 10, Hoermann's PTRS for lambda >= 10, 0 for lambda == 0, and stores the count + 1e-9
in the engine's precision.  The samplers here are the textbook spellings numpy's legacy generator
uses (`random_poisson_mult`, `random_poisson_ptrs`), vectorised over pixels with a per-pixel
lambda; the kernel evaluates the same inequalities in cheaper forms, so the two agree except when
a uniform falls within rounding of a decision boundary.  `explain_pixel` reports how far each
decision of one pixel was from its boundary, so that such a tie can be told apart from a wrong
counter or a lost write."""
import numpy as np
from scipy.special import gammaln

M32 = np.uint64(0xFFFFFFFF)


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    c0, c1, c2, c3 = (np.asarray(c, dtype=np.uint64) for c in (c0, c1, c2, c3))
    k0, k1 = np.uint64(k0), np.uint64(k1)
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c0
        p1 = np.uint64(0xCD9E8D57) * c2
        hi0, lo0, hi1, lo1 = p0 >> np.uint64(32), p0 & M32, p1 >> np.uint64(32), p1 & M32
        c0, c1, c2, c3 = hi1 ^ c1 ^ k0, lo1, hi0 ^ c3 ^ k1, lo0
        k0 = (k0 + np.uint64(0x9E3779B9)) & M32
        k1 = (k1 + np.uint64(0xBB67AE85)) & M32
    return c0, c1, c2, c3


def u01(hi, lo):
    return (((hi << np.uint64(32)) | lo) >> np.uint64(11)).astype(np.float64) * 2.0 ** -53


def counters(pixels, image, att, seed):
    """Philox output for counter (pixel lo, pixel hi, image, att), key = seed."""
    p = np.asarray(pixels).astype(np.uint64)
    zero = np.zeros_like(p)
    return philox4x32_10(p & M32, p >> np.uint64(32), zero + np.uint64(image), zero + np.uint64(att),
                         seed & 0xFFFFFFFF, seed >> 32)


def _ptrs_constants(lam):
    b = 0.931 + 2.53 * np.sqrt(lam)
    a = -0.059 + 0.02483 * b
    return a, b, 1.1239 + 1.1328 / (b - 3.4), 0.9277 - 3.6224 / (b - 2.0)


def textbook_ptrs(lam, seed, pixels, image=0):
    """numpy's legacy `random_poisson_ptrs` for lambda >= 10 (scalar or one per pixel), attempt
    `att` drawn from counter (pixel lo, pixel hi, image, att) with key = seed."""
    pixels = np.asarray(pixels)
    lam = np.broadcast_to(np.asarray(lam, dtype=np.float64), pixels.shape).ravel()
    pixels = pixels.ravel()
    out = np.full(pixels.size, -1.0)
    todo = np.arange(pixels.size)
    for att in range(64):
        if todo.size == 0:
            break
        lt = lam[todo]
        a, b, invalpha, vr = _ptrs_constants(lt)
        v = counters(pixels[todo], image, att, seed)
        U = u01(v[0], v[1]) - 0.5
        V = u01(v[2], v[3])
        us = 0.5 - np.abs(U)
        with np.errstate(divide='ignore', invalid='ignore'):
            k = np.floor((2.0 * a / us + b) * U + lt + 0.43)
            squeeze = (us >= 0.07) & (V <= vr)
            skip = (k < 0.0) | ((us < 0.013) & (V > us))
            exact = (np.log(V) + np.log(invalpha) - np.log(a / (us * us) + b)
                     <= -lt + k * np.log(lt) - gammaln(k + 1.0))
        accept = squeeze | (~skip & exact)
        out[todo[accept]] = k[accept]
        todo = todo[~accept]
    assert todo.size == 0
    return out


def textbook_multiplication(lam, seed, pixels, image=0):
    """Knuth's multiplication method (numpy's legacy `random_poisson_mult`) for lambda < 10
    (scalar or one per pixel): count uniforms until their product drops to exp(-lambda); each
    Philox call supplies two of them."""
    pixels = np.asarray(pixels).ravel()
    lam = np.broadcast_to(np.asarray(lam, dtype=np.float64), pixels.shape)
    enlam = np.exp(-lam)
    out = np.zeros(pixels.size)
    prod = np.ones(pixels.size)
    running = np.ones(pixels.size, dtype=bool)
    for att in range(200):
        idx = np.flatnonzero(running)
        if idx.size == 0:
            break
        v = counters(pixels[idx], image, att, seed)
        ua, ub = u01(v[0], v[1]), u01(v[2], v[3])
        prod[idx] *= ua
        done = ~(prod[idx] > enlam[idx])
        running[idx[done]] = False
        idx, ub = idx[~done], ub[~done]     # the second uniform: pixels still running only
        out[idx] += 1.0
        prod[idx] *= ub
        done = ~(prod[idx] > enlam[idx])
        running[idx[done]] = False
        out[idx[~done]] += 1.0
    assert not running.any()
    return out


def replay_counts(lam, seed, image):
    """Poisson counts of one image (any shape, pixel = flat index): 0 where lambda == 0,
    the multiplication method below 10, PTRS from 10 on."""
    lam = np.asarray(lam, dtype=np.float64)
    flat = lam.ravel()
    pixels = np.arange(flat.size, dtype=np.int64)
    counts = np.zeros(flat.size)
    small = (flat > 0.0) & (flat < 10.0)
    big = flat >= 10.0
    counts[small] = textbook_multiplication(flat[small], seed, pixels[small], image)
    counts[big] = textbook_ptrs(flat[big], seed, pixels[big], image)
    return counts.reshape(lam.shape)


def replay_field(noiseless, seed, image, dtype=np.float64):
    """What ROW_INV_SIM (and WIN_SIMULATE) store for image `image` whose noiseless values are
    `noiseless`: the count + 1e-9 rounded to the engine's precision `dtype`, as float64."""
    counts = replay_counts(noiseless, seed, image)
    return (counts + 1e-9).astype(dtype).astype(np.float64)


def explain_pixel(lam, seed, pixel, image):
    """Every decision the textbook sampler takes for one pixel, with its distance from the
    boundary (lines of text)."""
    lam = float(lam)
    lines = ['pixel %d image %d lambda %.17g' % (pixel, image, lam)]
    if not lam > 0.0:
        return lines + ['  lambda == 0: count 0']
    if lam < 10.0:
        enlam, prod, x = np.exp(-lam), 1.0, 0
        for att in range(200):
            v = counters(np.array([pixel]), image, att, seed)
            for u in (u01(v[0], v[1])[0], u01(v[2], v[3])[0]):
                prod *= u
                lines.append('  attempt %d: count %d, product / exp(-lambda) - 1 = %.3e'
                             % (att, x, prod / enlam - 1.0))
                if not prod > enlam:
                    return lines
                x += 1
        return lines
    a, b, invalpha, vr = _ptrs_constants(lam)
    for att in range(64):
        v = counters(np.array([pixel]), image, att, seed)
        U = u01(v[0], v[1])[0] - 0.5
        V = u01(v[2], v[3])[0]
        us = 0.5 - abs(U)
        arg = (2.0 * a / us + b) * U + lam + 0.43
        k = np.floor(arg)
        msg = ('  attempt %d: k %d, floor argument %.3e from an integer, squeeze us - 0.07 = %.3e'
               ' V - v_r = %.3e' % (att, k, min(arg - k, k + 1 - arg), us - 0.07, V - vr))
        if us >= 0.07 and V <= vr:
            lines.append(msg + ' -> squeeze accepts')
            return lines
        if k < 0 or (us < 0.013 and V > us):
            lines.append(msg + ' -> skipped')
            continue
        lhs = np.log(V) + np.log(invalpha) - np.log(a / (us * us) + b)
        rhs = -lam + k * np.log(lam) - gammaln(k + 1.0)
        lines.append(msg + ', exact test lhs - rhs = %.3e -> %s'
                     % (lhs - rhs, 'accepts' if lhs <= rhs else 'rejects'))
        if lhs <= rhs:
            return lines
    return lines


def assert_field(got, noiseless, seed, image, dtype, show=4):
    """`got` (one image) must equal replay_field(noiseless, seed, image, dtype) in every pixel;
    the message names the first mismatching pixels and explains their draws."""
    got = np.asarray(got, dtype=np.float64).reshape(np.shape(noiseless))
    want = replay_field(noiseless, seed, image, dtype)
    bad = np.flatnonzero(got.ravel() != want.ravel())
    if bad.size == 0:
        return
    lam = np.asarray(noiseless, dtype=np.float64).ravel()
    lines = ['%d of %d pixels differ from the textbook field (image %d, seed %d)'
             % (bad.size, got.size, image, seed)]
    for p in bad[:show]:
        lines.append('pixel %d (y, x) = %s: got %.17g, want %.17g'
                     % (p, np.unravel_index(p, got.shape), got.ravel()[p], want.ravel()[p]))
        lines += explain_pixel(lam[p], seed, int(p), image)
    raise AssertionError('\n'.join(lines))
