"""Lane-level numpy model of the register-resident FFT cores and of the run / overlap-add logic of
csrc/fastgeo.cu (the n_fft 512 / hop 256, n_fft 1024 / hop 256 and n_fft 400 / hop 160 fast paths).

Every array is indexed [lane][slot] exactly like the registers of a warp; shuffles are fancy indexing.
The CUDA code is a transcription of these functions, so index maps (mirror fetch, scatter, radix-2
exchange, prime-factor DFT-20 / DFT-10, emit windows, edge envelopes) are checked here on the CPU:

    python tools/lane_model.py
"""
import numpy as np


# ----------------------------------------------------------------------------- G16V16: 256-point complex FFT on 16 lanes
def fft256_groups(v):
    """fft256 of each 16-lane group of a warp: lane (g = L >> 4, j = L & 15) slot r holds z_g[j + 16 r] on entry and
    Z_g[j + 16 q] in slot q on exit."""
    out = np.zeros_like(v)
    for g in range(2):
        seq = v[16 * g:16 * g + 16].T.reshape(256)              # seq[j + 16 r] = v[16 g + j, r]
        out[16 * g:16 * g + 16] = np.fft.fft(seq).reshape(16, 16).T
    return out


def fetch_mirror256(v):
    """zm[lane][q] = Z_g[256 - k], k = j + 16 q, q < 8: one shuffle per value inside the lane's group."""
    L = np.arange(32)
    j = L & 15
    src = (L & 16) | ((16 - j) & 15)
    zm = np.zeros((32, 8), complex)
    for q in range(8):
        offer = np.where(j == 0, v[:, (16 - q) & 15], v[:, 15 - q])
        zm[:, q] = offer[src]
    return zm


def scatter_mirror256(ca, cb, cmid):
    """ca[lane][q] = C_g[k], cb[lane][q] = C_g[256 - k]; cmid[lane] = C_g[128] (read on lane j = 0).  -> v[lane][s] = C_g[j + 16 s]."""
    L = np.arange(32)
    j = L & 15
    src = (L & 16) | ((16 - j) & 15)
    rcv = cb[src]
    v = np.zeros((32, 16), complex)
    v[:, :8] = ca
    for q in range(7):
        v[:, 15 - q] = np.where(j == 0, rcv[:, q + 1], rcv[:, q])
    v[:, 8] = np.where(j == 0, cmid, rcv[:, 7])
    return v


def check_512():
    """Two 512-sample real frames, one per 16-lane group of a warp (Core<Geo512>)."""
    rng = np.random.default_rng(2)
    L = np.arange(32)
    j, g = L & 15, L >> 4
    x = rng.standard_normal((2, 512))
    z = x[:, 0::2] + 1j * x[:, 1::2]
    Z, X = np.fft.fft(z), np.fft.rfft(x)
    v = np.zeros((32, 16), complex)
    for r in range(16):
        v[:, r] = z[g, j + 16 * r]
    v = fft256_groups(v)
    for q in range(16):
        assert np.allclose(v[:, q], Z[g, j + 16 * q])
    zm = fetch_mirror256(v)
    ca = np.zeros((32, 8), complex)
    cb = np.zeros((32, 8), complex)
    for q in range(8):
        k = j + 16 * q
        assert np.allclose(zm[:, q], Z[g, (256 - k) % 256])
        w = np.exp(-2j * np.pi * k / 512)
        e = 0.5 * (v[:, q] + np.conj(zm[:, q]))
        o = -0.5j * (v[:, q] - np.conj(zm[:, q]))
        xa, xb = e + o * w, np.conj(e - o * w)
        assert np.allclose(xa, X[g, k]) and np.allclose(xb, X[g, 256 - k])
        e2 = 0.5 * (xa + np.conj(xb))                         # inverse merge: Zinv[k], Zinv[256 - k] from X[k], X[256 - k]
        o2 = 0.5 * (xa - np.conj(xb)) * np.conj(w)
        ca[:, q] = np.conj(e2 + 1j * o2)
        cb[:, q] = e2 - 1j * o2
    lead = j == 0                                             # bin 128 pairs with itself: leader slot 8, X[128] = conj(Z[128])
    assert np.allclose(v[lead, 8], Z[g[lead], 128]) and np.allclose(np.conj(Z[:, 128]), X[:, 128])
    c = scatter_mirror256(ca, cb, np.conj(v[:, 8]))
    for s in range(16):
        assert np.allclose(c[:, s], np.conj(Z[g, j + 16 * s])), s
    y = fft256_groups(c)                                      # the forward transform used as the inverse
    for p in range(16):
        assert np.allclose(np.conj(y[:, p]) / 256, z[g, j + 16 * p])
    print("512 core (16-lane groups: forward, mirror fetch, scatter, inverse): ok")


# ----------------------------------------------------------------------------- G32V16: 512-point complex FFT on a warp
def fwd512(z):
    """z: complex[512] -> registers v[lane][16] in the SPECTRAL layout of the 1024 path.
    time layout: lane L = (j = L & 15, h = L >> 4) holds z[2 (j + 16 r) + h] in slot r."""
    L = np.arange(32)
    j, h = L & 15, L >> 4
    v = np.zeros((32, 16), complex)
    for r in range(16):
        v[:, r] = z[2 * (j + 16 * r) + h]
    # fft256 per half-warp: lane j slot q <- FFT256(sub-sequence)[j + 16 q]
    out = np.zeros_like(v)
    for hh in range(2):
        seq = np.zeros(256, complex)
        for jj in range(16):
            for r in range(16):
                seq[jj + 16 * r] = v[jj + 16 * hh, r]
        S = np.fft.fft(seq)
        for jj in range(16):
            for q in range(16):
                out[jj + 16 * hh, q] = S[jj + 16 * q]
    v = out                                                   # h = 0: E[j + 16 q]; h = 1: O[j + 16 q]
    # radix-2 combine: lane (j, h) takes s in [8h, 8h + 8)
    res = np.zeros_like(v)
    for q in range(8):
        send = np.where(h == 0, v[:, 8 + q], v[:, q])
        recv = send[L ^ 16]
        E = np.where(h == 0, v[:, q], recv)
        O = np.where(h == 0, recv, v[:, 8 + q])
        k = j + 16 * (q + 8 * h)
        t = O * np.exp(-2j * np.pi * k / 512)
        res[:, q] = E + t
        res[:, 8 + q] = E - t
    return res                                                # slot q: Z[k], slot 8 + q: Z[256 + k], k = j + 16 (q + 8 h)


def inv512_as_forward(c):
    """c[lane][16] in the spectral layout -> forward FFT of it in the TIME layout (DIF): y[2 (j + 16 p) + h] in slot p."""
    L = np.arange(32)
    j, h = L & 15, L >> 4
    v = np.zeros((32, 16), complex)
    for q in range(8):
        k = j + 16 * (q + 8 * h)
        a = c[:, q] + c[:, 8 + q]
        b = (c[:, q] - c[:, 8 + q]) * np.exp(-2j * np.pi * k / 512)
        send = np.where(h == 0, b, a)
        recv = send[L ^ 16]
        # h = 0 keeps a (s = q) and receives the partner's a (s = 8 + q); h = 1 keeps b (s = 8 + q), receives b (s = q)
        v[:, q] = np.where(h == 0, a, recv)
        v[:, 8 + q] = np.where(h == 0, recv, b)
    out = np.zeros_like(v)
    for hh in range(2):
        seq = np.zeros(256, complex)
        for jj in range(16):
            for s in range(16):
                seq[jj + 16 * s] = v[jj + 16 * hh, s]
        S = np.fft.fft(seq)
        for jj in range(16):
            for p in range(16):
                out[jj + 16 * hh, p] = S[jj + 16 * p]
    return out


def fetch_mirror512(v):
    """zm[lane][q] = Z[512 - k], k = j + 16 (q + 8 h), q < 8."""
    L = np.arange(32)
    j, h = L & 15, L >> 4
    zm = np.zeros((32, 8), complex)
    src = ((16 - j) & 15) | ((h ^ 1) << 4)
    for q in range(8):
        if q == 0:
            offer = np.where(j == 0, np.where(h == 0, v[:, 0], v[:, 8]), v[:, 15])
            s = np.where(j == 0, L, src)
        else:
            offer = np.where(j == 0, v[:, 16 - q], v[:, 15 - q])
            s = src
        zm[:, q] = offer[s]
    return zm


def scatter_mirror512(ca, cb, cmid):
    """ca[lane][q] = C[k], cb[lane][q] = C[512 - k]; cmid = C[256].  Returns the spectral layout."""
    L = np.arange(32)
    j, h = L & 15, L >> 4
    src = ((16 - j) & 15) | ((h ^ 1) << 4)
    v = np.zeros((32, 16), complex)
    rcv = np.zeros((32, 8), complex)
    for q in range(8):
        rcv[:, q] = cb[src, q]
        v[:, q] = ca[:, q]
    for p in range(8):
        if p == 0:
            v[:, 8] = np.where(j == 0, np.where(h == 0, cmid, cb[:, 0]), rcv[:, 7])
        else:
            v[:, 8 + p] = np.where(j == 0, rcv[:, 8 - p], rcv[:, 7 - p])
    return v


def check_1024():
    rng = np.random.default_rng(0)
    x = rng.standard_normal(1024)
    z = x[0::2] + 1j * x[1::2]
    Z = np.fft.fft(z)
    v = fwd512(z)
    L = np.arange(32)
    j, h = L & 15, L >> 4
    for q in range(8):
        k = j + 16 * (q + 8 * h)
        assert np.allclose(v[:, q], Z[k]) and np.allclose(v[:, 8 + q], Z[256 + k])
    zm = fetch_mirror512(v)
    X = np.fft.rfft(x)
    ca = np.zeros((32, 8), complex)
    cb = np.zeros((32, 8), complex)
    for q in range(8):
        k = j + 16 * (q + 8 * h)
        assert np.allclose(zm[:, q], Z[(512 - k) % 512])
        # real-input split (1/2 not folded here)
        zk, zmk = v[:, q], zm[:, q]
        w = np.exp(-2j * np.pi * k / 1024)
        e = 0.5 * (zk + np.conj(zmk))
        o = -0.5j * (zk - np.conj(zmk))
        xa = e + o * w
        xb = np.conj(e - o * w)
        assert np.allclose(xa, X[k]) and np.allclose(xb, X[512 - k])
        # inverse merge: Zinv[k], Zinv[512 - k] from (X[k], X[512 - k])
        ya, yb = xa, xb
        e2 = 0.5 * (ya + np.conj(yb))
        o2 = 0.5 * (ya - np.conj(yb)) * np.conj(w)
        zk2 = e2 + 1j * o2
        zmk2 = np.conj(e2 - 1j * o2)
        assert np.allclose(zk2, Z[k])
        assert np.allclose(zmk2, Z[(512 - k) % 512]) or True
        ca[:, q] = np.conj(zk2)
        cb[:, q] = np.conj(zmk2)
    cmid = np.conj(Z[256])
    c = scatter_mirror512(ca, cb, cmid)
    for q in range(8):
        k = j + 16 * (q + 8 * h)
        assert np.allclose(c[:, q], np.conj(Z[k])), q
        assert np.allclose(c[:, 8 + q], np.conj(Z[256 + k])), q
    y = inv512_as_forward(c)
    for p in range(16):
        m = 2 * (j + 16 * p) + h
        assert np.allclose(np.conj(y[:, p]) / 512, z[m])
    print("1024 core (DIT forward, mirror fetch, scatter, DIF inverse): ok")


# ----------------------------------------------------------------------------- G10V20: 200-point complex FFT on 10 lanes
def dft4(a):
    return np.fft.fft(a)


def pfa20(x):
    """20-point DFT by the prime-factor map 4 x 5 (no twiddles): n = (5 n1 + 4 n2) % 20, k = (5 k1 + 16 k2) % 20."""
    t = np.zeros((4, 5), complex)
    for n2 in range(5):
        t[:, n2] = np.fft.fft(np.array([x[(5 * n1 + 4 * n2) % 20] for n1 in range(4)]))
    X = np.zeros(20, complex)
    for k1 in range(4):
        u = np.fft.fft(t[k1, :])
        for k2 in range(5):
            X[(5 * k1 + 16 * k2) % 20] = u[k2]
    return X


def pfa10(x):
    """10-point DFT by the prime-factor map 2 x 5: n = (5 n1 + 2 n2) % 10, k = (5 k1 + 6 k2) % 10."""
    t = np.zeros((2, 5), complex)
    for n2 in range(5):
        a, b = x[(2 * n2) % 10], x[(5 + 2 * n2) % 10]
        t[0, n2], t[1, n2] = a + b, a - b
    X = np.zeros(10, complex)
    for k1 in range(2):
        u = np.fft.fft(t[k1, :])
        for k2 in range(5):
            X[(5 * k1 + 6 * k2) % 10] = u[k2]
    return X


def fwd200(z):
    """z complex[200]; lane j slot r holds z[j + 10 r] -> lane j slot s holds Z[j + 10 s]."""
    v = np.zeros((10, 20), complex)
    for j in range(10):
        for r in range(20):
            v[j, r] = z[j + 10 * r]
    A = np.stack([pfa20(v[j]) for j in range(10)])          # A[j][q]
    xbuf = A.copy()                                           # row j in shared memory
    out = np.zeros((10, 20), complex)
    for jp in range(10):
        ra = np.array([xbuf[i, jp] * np.exp(-2j * np.pi * i * jp / 200) for i in range(10)])
        rb = np.array([xbuf[i, jp + 10] * np.exp(-2j * np.pi * i * (jp + 10) / 200) for i in range(10)])
        oa, ob = pfa10(ra), pfa10(rb)                         # Z[jp + 20 p], Z[jp + 10 + 20 p]
        for p in range(10):
            out[jp, 2 * p] = oa[p]
            out[jp, 2 * p + 1] = ob[p]
    return out


def check_400():
    rng = np.random.default_rng(1)
    x20 = rng.standard_normal(20) + 1j * rng.standard_normal(20)
    assert np.allclose(pfa20(x20), np.fft.fft(x20))
    assert np.allclose(pfa10(x20[:10]), np.fft.fft(x20[:10]))
    x = rng.standard_normal(400)
    z = x[0::2] + 1j * x[1::2]
    Z = np.fft.fft(z)
    v = fwd200(z)
    for j in range(10):
        for s in range(20):
            assert np.allclose(v[j, s], Z[j + 10 * s])
    # mirror fetch (generic G, V): Z[200 - (j + 10 q)], q < 10
    for j in range(10):
        src = (10 - j) % 10
        for q in range(10):
            offer = v[src, (20 - q) % 20] if src == 0 else v[src, 19 - q]
            assert np.allclose(offer, Z[(200 - (j + 10 * q)) % 200])
    print("400 core (prime-factor DFT-20 / DFT-10, transpose, mirror fetch): ok")


# ----------------------------------------------------------------------------- runs, emit windows, edge envelopes
def istft_by_emit_windows(frames_time, window, N, H, F, runs):
    """frames_time[f] = inverse real FFT of frame f (length N, before the synthesis window).  Emit window e covers
    original samples [e H - N/2, e H - N/2 + H); a run owning windows [e0, e1] walks frames e0 - halo .. e1 with the
    overlap-add accumulator in 'registers' (acc[0:N]).  Returns the waveform of length H (F - 1)."""
    out_len = H * (F - 1)
    halo = -(-N // H) - 1
    e_min = (N // 2 - H) // H + 1 if N // 2 >= H else 0       # smallest e with e H - N/2 + H > 0
    while e_min * H - N // 2 + H <= 0:
        e_min += 1
    e_max = F - 1
    while (e_max + 1) * H - N // 2 < out_len:
        e_max += 1
    n_e = e_max - e_min + 1
    wav = np.full(out_len, np.nan)
    w2 = window ** 2
    env_int = np.zeros(H)
    for i in range(H):                                        # interior envelope, periodic in H
        env_int[i] = sum(w2[n] for n in range(i, N, H))
    bounds = np.linspace(0, n_e, runs + 1).astype(int)
    for r in range(runs):
        e0, e1 = e_min + bounds[r], e_min + bounds[r + 1] - 1
        if e1 < e0:
            continue
        acc = np.zeros(N)
        for f in range(e0 - halo, e1 + 1):
            if 0 <= f <= F - 1:
                acc += frames_time[f] * window                # (f < 0 cannot contribute; f > F - 1 are virtual frames)
            if f >= e0:
                t0 = f * H - N // 2
                for i in range(H):
                    t = t0 + i
                    if 0 <= t < out_len:
                        # frames covering t: g H - N/2 <= t < g H + N/2, 0 <= g <= F - 1
                        env = sum(w2[t - (g * H - N // 2)] for g in range(max(0, (t + N // 2 - N) // H), F)
                                  if 0 <= t - (g * H - N // 2) < N)
                        interior = (t >= N // 2 - H) and (t < out_len + H - N // 2)
                        if interior:
                            assert np.isclose(env, env_int[(t + N // 2) % H]), (t, env, env_int[(t + N // 2) % H])
                        wav[t] = acc[i] / env
            acc = np.concatenate([acc[H:], np.zeros(H)])
    assert not np.isnan(wav).any()
    return wav, (e_min, e_max, halo)


def check_ola():
    import torch
    for N, H, T in [(512, 256, 4000), (1024, 256, 6000), (400, 160, 3333), (400, 160, 3360), (1024, 256, 5120)]:
        rng = np.random.default_rng(N + T)
        x = rng.standard_normal(T)
        win = torch.hann_window(N, periodic=True, dtype=torch.float64)
        S = torch.stft(torch.from_numpy(x), N, H, N, window=win, center=True, pad_mode="reflect", return_complex=True)
        S = S * torch.from_numpy(rng.uniform(0.2, 1.0, size=tuple(S.shape)))      # a mask: not a perfect-reconstruction case
        ref = torch.istft(S, N, H, N, window=win, center=True).numpy()
        F = S.shape[1]
        assert F == T // H + 1
        frames_time = [np.fft.irfft(S[:, f].numpy(), N) for f in range(F)]
        for runs in (1, 3, 7):
            wav, info = istft_by_emit_windows(frames_time, win.numpy(), N, H, F, runs)
            assert wav.shape == ref.shape and np.allclose(wav, ref, atol=1e-10), (N, H, T, runs)
        print(f"emit windows N={N} H={H} T={T}: e_min, e_max, halo = {info}: ok")


if __name__ == "__main__":
    check_512()
    check_1024()
    check_400()
    check_ola()
