"""Cast / per-band normalise / one-hot / band statistics (oracle; test infrastructure only).

North-star row A17 (SURVEY.md section 8a) — NOT in the reference (its nearest analogue is display scaling by
the per-band max, ``parse_tfrecords.ipynb`` cell 21), so **parity is unpinned**; the definition is:

    x_hat[n,y,x,b]  = (float32(x) - mean[b]) / std[b]           float32 arithmetic, IEEE division
    onehot[n,y,x,k] = 1.0f if label == k else 0.0f,  k in [0,K) (tf.one_hot: out-of-range -> all zero)
    stats per band  = n, sum x, sum x^2 over valid pixels, exact integers;
                      mean/std derived in float64 then cast to float32.
"""
import numpy as np


def normalise(img, mean, std):
    img = np.asarray(img)
    mean = np.asarray(mean, dtype=np.float32)
    std = np.asarray(std, dtype=np.float32)
    return (img.astype(np.float32) - mean) / std


def one_hot(label, num_classes):
    label = np.asarray(label)
    if label.ndim and label.shape[-1] == 1 and label.ndim == 3:
        label = label[..., 0]
    # value equality, no cast: a float label that is NaN, infinite, negative or not integral is no class
    k = np.arange(num_classes, dtype=np.int64)
    return (label[..., None] == k).astype(np.float32)


def band_stats(img, valid=None):
    """-> int array (B,3): n, sum, sumsq as Python ints (object dtype) — exact."""
    img = np.asarray(img)
    B = img.shape[-1]
    out = []
    v = None if valid is None else (np.asarray(valid).reshape(-1) != 0)
    x = img.reshape(-1, B)
    if v is not None:
        x = x[v]
    for b in range(B):
        col = x[:, b].astype(np.int64)
        n = int(col.size)
        s = int(col.sum(dtype=np.int64))
        # x^2 up to 2^32, count up to 2^31 here: split to stay exact in int64
        sq = col * col
        ss = int((sq >> 16).sum(dtype=np.int64)) * 65536 + int((sq & 0xFFFF).sum(dtype=np.int64))
        out.append((n, s, ss))
    return out


def mean_std_from_stats(stats):
    """Exact integer stats -> (mean, std) float32 arrays via float64 (population std)."""
    mean, std = [], []
    for n, s, ss in stats:
        if n == 0:
            mean.append(0.0)
            std.append(1.0)
            continue
        # exact rationals, one correctly-rounded division each (Python int / int)
        mean.append(s / n)
        std.append(((ss * n - s * s) / (n * n)) ** 0.5)
    return np.asarray(mean, dtype=np.float64).astype(np.float32), np.asarray(std, dtype=np.float64).astype(np.float32)
