"""Generate the golden fixtures under tests/golden/ from the REFERENCE ITSELF.

Runs only in the build container (needs /root/reference): it drives oracle/_ref/libwsref.so, i.e. the
reference's own src/scene/WSTessendorf.cpp compiled verbatim (oracle/Makefile), with srand(seed) fixed,
FFT behind the FFTW-API shim evaluated in float64.  The reference has no tests or golden vectors of
its own for this path (SURVEY.md §4), so these files are the pinned outputs of the reference code.

    python tests/golden/make_golden.py

Each case -> params, seed, xi (Gaussian array), h0 (N,N,5 fp32: the reference's 20-byte record), wave_vectors,
t[], A[], minh[], maxh[], disp[t], norm[t], and (small N) the pre-FFT spectra, packed into <name>.npz, <name>.1.npz, ...
so that every file stays under 1 MB (tests/conftest.py load_golden() merges them).
"""
import io
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import refmodel as R  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
PART_BYTES = 990_000   # bytes per file (each array measured as its own .npz, headers included): below 1 MB


def _compressed_size(key, a):
    buf = io.BytesIO()
    np.savez_compressed(buf, **{key: a})
    return buf.tell()


def save_case(name, arrays):
    """Pack the arrays of one case, in order, into as few files of at most PART_BYTES as fit."""
    parts, size = [{}], 0
    for key, a in arrays.items():
        n = _compressed_size(key, a)
        if n > PART_BYTES:
            raise ValueError(f"{name}/{key}: {n} bytes compressed does not fit one file")
        if parts[-1] and size + n > PART_BYTES:
            parts.append({})
            size = 0
        parts[-1][key] = a
        size += n
    for f in os.listdir(OUT):
        if f.startswith(name + ".") and f.endswith(".npz"):
            os.remove(os.path.join(OUT, f))
    for i, part in enumerate(parts):
        path = os.path.join(OUT, name + (f".{i}" if i else "") + ".npz")
        np.savez_compressed(path, **part)
        print(path, os.path.getsize(path) // 1024, "KiB")


CASES = [
    # name, N, L, wind, V, A, damping, T, lambda, seed, times, with_spectra
    ("n16_default", 16, 1000.0 * 16 / 512, (1.0, 1.0), 30.0, 3e-7, 0.1, 200.0, -1.0, 1234,
     [0.0, 1.5, 100.0, 10000.25], True),
    ("n64_default", 64, 1000.0 * 64 / 512, (1.0, 1.0), 30.0, 3e-7, 0.1, 200.0, -1.0, 1234,
     [0.0, 1.5, 100.0, 1234.567], True),
    ("n64_wind", 64, 300.0, (-0.4, 1.7), 11.0, 5e-7, 0.25, 120.0, -0.6, 77,
     [0.0, 33.25], True),
    ("n256_default", 256, 1000.0 * 256 / 512, (1.0, 1.0), 30.0, 3e-7, 0.1, 200.0, -1.0, 1234,
     [777.77], False),
]


def main():
    for (name, n, L, wind, V, A, damp, T, lam, seed, times, with_spec) in CASES:
        m = R.RefWSTessendorf(n, L, fft_mode=R.FFT_FLOAT64)
        m.SetWindDirection(*wind)
        m.SetWindSpeed(V)
        m.SetPhillipsConst(A)
        m.SetDamping(damp)
        m.SetAnimationPeriod(T)
        m.SetLambda(lam)
        xi = m.GaussArray(seed)
        m.Prepare(seed)
        h0 = m.ExportH0()
        wv = m.ExportWaveVectors()
        out = dict(
            params=np.array([n, L, wind[0], wind[1], V, A, damp, T, lam], np.float64),
            seed=np.int64(seed), xi=xi,
            h0=np.stack([h0[f] for f in h0.dtype.names], axis=-1),
            wave_vectors=wv, t=np.array(times, np.float32))
        As, mins, maxs, disps, norms, specs = [], [], [], [], [], []
        for t in times:
            if with_spec:
                R.lib().wsref_set_fft_mode(R.FFT_NOOP)
                m.ComputeWaves(t)
                specs.append(m.ExportWorkArrays())
                R.lib().wsref_set_fft_mode(R.FFT_FLOAT64)
            As.append(m.ComputeWaves(t))
            mins.append(m.GetMinHeight())
            maxs.append(m.GetMaxHeight())
            disps.append(m.GetDisplacements())
            norms.append(m.GetNormals())
        out.update(A=np.array(As, np.float32), minh=np.array(mins, np.float32),
                   maxh=np.array(maxs, np.float32), disp=np.stack(disps), norm=np.stack(norms))
        if with_spec:
            out["spectra"] = np.stack(specs)
        save_case(name, out)


if __name__ == "__main__":
    main()
