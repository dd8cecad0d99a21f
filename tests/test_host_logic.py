"""CPU-only checks of host-side logic that the GPU kernels rely on, and of bench.py's reference-arm contract line."""
import json
import os
import subprocess
import sys

import numpy as np

from oracle import dl4j_oracle as o

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def pack_deconv_ps(w_int, O, C):
    """NumPy mirror of pack_deconv_ps_kernel (kernels_tc.cu): w_int [O][4][4][C] -> wps [(py,px,c4)][(dyr,dxc)][O]."""
    wps = np.zeros((16, 9, O), w_int.dtype)
    for py in range(2):
        for px in range(2):
            for c in range(C):
                n = (py * 2 + px) * 4 + c
                for t in range(9):
                    dyr, dxc = t // 3 - 1, t % 3 - 1
                    r = {(-1, 0): 3, (0, 0): 1, (0, 1): 2, (1, 1): 0}.get((dyr, py), -1)
                    s = {(-1, 0): 3, (0, 0): 1, (0, 1): 2, (1, 1): 0}.get((dxc, px), -1)
                    if r >= 0 and s >= 0:
                        wps[n, t, :] = w_int[:, r, s, c]
    return wps


def test_pixel_shuffle_form_of_the_transposed_conv_equals_deconvolution2d():
    """The tcgen05 G-last forward computes ONE 3x3 s1 p1 conv with 16 = (py,px,c4) output columns over the deconv input and scatters
    each pixel's 16 values to its 2x2 output block.  With the packed weights this must equal Deconvolution2D 4x4 s2 p1 (J:203-219 family)."""
    rng = np.random.default_rng(0)
    n, O, C, h = 2, 8, 3, 5                                  # deconv: O input channels on an h x h grid -> C channels on 2h x 2h
    dec = o.Deconv2D(O, C, (4, 4), (2, 2), (1, 1), has_bias=False); dec.init(rng, np.float64)
    x = rng.standard_normal((n, O, h, h))
    want = dec.forward(x, True)                              # [n, C, 2h, 2h]
    # internal weight layout of the engine for this layer: [O][taps][C] (conv-equivalent geometry: g.O = deconv nIn, g.C = deconv nOut)
    w_int = dec.params["W"].transpose(0, 2, 3, 1)            # [nIn=O][kh][kw][nOut=C]
    wps = pack_deconv_ps(w_int, O, C)                        # [16][9][O]
    conv = o.Conv2D(O, 16, (3, 3), (1, 1), (1, 1), has_bias=False); conv.init(rng, np.float64)
    conv.params["W"] = wps.reshape(16, 3, 3, O).transpose(0, 3, 1, 2).copy()      # [16][O][3][3]
    y16 = conv.forward(x, True)                              # [n, 16, h, h]
    got = np.zeros_like(want)
    for py in range(2):
        for px in range(2):
            for c in range(C):
                got[:, c, py::2, px::2] = y16[:, (py * 2 + px) * 4 + c]
    np.testing.assert_allclose(got, want, rtol=1e-12, atol=1e-12)
    # the padded channel slots stay zero
    for py in range(2):
        for px in range(2):
            assert np.all(y16[:, (py * 2 + px) * 4 + 3] == 0)


def test_edge_im2col_row_layout():
    """tc_edge_conv builds, per output pixel, the row k = (r*4+s)*C + c from the 4 x (4*C) window starting at input (2oy-1, 2ox-1):
    the same K ordering as the engine's weight rows [O][16 taps][C], so out = rows @ W_int^T must equal ConvolutionLayer 4x4 s2 p1."""
    rng = np.random.default_rng(1)
    n, C, O, H = 2, 3, 5, 8
    conv = o.Conv2D(C, O, (4, 4), (2, 2), (1, 1), has_bias=False); conv.init(rng, np.float64)
    x = rng.standard_normal((n, C, H, H)); want = conv.forward(x, True)
    xh = np.pad(x.transpose(0, 2, 3, 1), ((0, 0), (1, 1), (1, 1), (0, 0)))          # NHWC with the zero border
    w_int = conv.params["W"].transpose(0, 2, 3, 1).reshape(O, 16 * C)              # [O][(r,s,c)]
    got = np.zeros((n, H // 2, H // 2, O))
    for oy in range(H // 2):
        for ox in range(H // 2):
            rows = xh[:, 2 * oy:2 * oy + 4, 2 * ox:2 * ox + 4, :].reshape(n, 16 * C)   # k = (r*4+s)*C + c
            got[:, oy, ox] = rows @ w_int.T
    np.testing.assert_allclose(got.transpose(0, 3, 1, 2), want, rtol=1e-12, atol=1e-12)


def test_bench_reference_arm_prints_the_contract_line():
    env = dict(os.environ)          # default engine: oracle/cpu_ref.c (the C + OpenMP restatement of the DL4J CPU algorithm)
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", "c5", "--steps", "2", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, env=env)
    assert out.returncode == 0, out.stderr[-500:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert line["impl"] == "reference" and line["steps"] == 2 and line["warmup"] == 1 and line["higher_is_better"] is True
    for k in ("metric", "value", "unit", "n_gpus", "ms_per_step", "scaling", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in line, k
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["value"] == line["value"] and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["value"] > 0


def test_bench_dump_outputs_stay_under_budget_and_repeat(tmp_path):
    """bench.py --dump-outputs: small arrays are written whole, large ones share the byte budget as seeded samples that repeat run to run."""
    import bench
    arrays = {"losses": np.array([0.5, -1.0, 2.0]), "a": np.arange(400_000, dtype=np.float64), "b": -np.arange(300_000)}
    for d in ("x", "y"):
        bench.dump_outputs(str(tmp_path / d), arrays, budget=1_000_000)
    got = {k: np.load(tmp_path / "x" / f"{k}.npy") for k in arrays}
    assert all(v.dtype == np.float32 and v.ndim == 1 for v in got.values())
    assert np.array_equal(got["losses"], arrays["losses"])
    assert sum(v.nbytes for v in got.values()) <= 1_000_000 and got["a"].size > got["b"].size > 0
    assert np.all(np.diff(got["a"]) > 0) and np.isin(got["a"], arrays["a"]).all()           # sorted sample of the original elements
    for k in arrays:
        assert np.array_equal(got[k], np.load(tmp_path / "y" / f"{k}.npy")), k
    bench.dump_outputs(str(tmp_path / "z"), {"a": arrays["a"]}, budget=10_000_000)
    assert np.array_equal(np.load(tmp_path / "z" / "a.npy"), arrays["a"])                   # under the budget: written whole


def test_checkpoint_container_round_trip_and_nd4j_stream_layout(tmp_path):
    """ModelSerializer-style zip (J:606-618): round trip, and the byte layout of the ND4J stream restated in serializer.py."""
    import io
    import struct
    import zipfile
    from gan_deeplearning4j_b200 import serializer as sz, models as m
    rng = np.random.default_rng(0)
    specs = m.dcgan_discriminator(16, 8, 3)
    p = rng.standard_normal(1234).astype(np.float32); u = rng.standard_normal(2468).astype(np.float32)

    class FakeNet:            # the part of the Net interface the wrappers use
        def __init__(self): self.p, self.u = p.copy(), u.copy()
        def params(self): return self.p
        def updater_state(self): return self.u
        def num_params(self): return self.p.size
        def set_params(self, v): self.p = np.asarray(v, np.float32).copy()
        def set_updater_state(self, v): self.u = np.asarray(v, np.float32).copy()
    path = tmp_path / "dis.zip"
    sz.save_net(FakeNet(), path, specs, (3, 16, 16), meta={"precision": "bf16", "iteration": 7})
    with zipfile.ZipFile(path) as z:
        assert {"configuration.json", "coefficients.bin", "updaterState.bin"} <= set(z.namelist())        # DL4J's entry names
        raw = z.read("coefficients.bin")
    # shape-info buffer: writeUTF("LONG_SHAPE") writeLong(8) writeUTF("LONG") {2,1,n,n,1,0,1,'c'}; data: writeUTF writeLong(n) writeUTF("FLOAT") big-endian floats
    b = io.BytesIO(raw)
    assert b.read(2) == struct.pack(">H", 10) and b.read(10) == b"LONG_SHAPE" and struct.unpack(">q", b.read(8))[0] == 8
    assert b.read(2) == struct.pack(">H", 4) and b.read(4) == b"LONG"
    assert list(struct.unpack(">8q", b.read(64))) == [2, 1, 1234, 1234, 1, 0, 1, 99]
    assert b.read(2 + 10) == struct.pack(">H", 10) + b"LONG_SHAPE" and struct.unpack(">q", b.read(8))[0] == 1234
    assert b.read(2 + 5) == struct.pack(">H", 5) + b"FLOAT"
    assert struct.unpack(">f", b.read(4))[0] == p[0]
    other = FakeNet(); other.p[:] = 0; other.u[:] = 0
    got = sz.restore_into(other, path)
    assert np.array_equal(other.p, p) and np.array_equal(other.u, u) and got["meta"]["iteration"] == 7 and got["input_shape"] == (3, 16, 16)
    assert [l["type"] for l in got["specs"]] == [l["type"] for l in specs]
    sz.save_net(FakeNet(), path, specs, (3, 16, 16), save_updater=False)
    assert sz.read_model(path)["updater_state"] is None
    # a legacy (int-length) header is still readable
    legacy = io.BytesIO(); legacy.write(struct.pack(">H", 4) + b"HEAP" + struct.pack(">i", 8) + struct.pack(">H", 3) + b"INT" + np.array([2, 1, 3, 3, 1, 0, 1, 99], ">i4").tobytes())
    legacy.write(struct.pack(">H", 4) + b"HEAP" + struct.pack(">i", 3) + struct.pack(">H", 5) + b"FLOAT" + np.array([1, 2, 3], ">f4").tobytes()); legacy.seek(0)
    assert np.array_equal(sz.read_nd4j_array(legacy), np.array([[1, 2, 3]], np.float32))


def test_peer_memory_allreduce_slicing_and_sum_order():
    """Index arithmetic of p2p_allreduce_kernel (kernels_ew.cu) restated: the 16-byte vectors of the gradient are cut into W slices, rank r reduces
    slice r from every peer in rank order and writes it back to every peer; the n % 4 tail belongs to the last rank.  Every element must have
    exactly one reader-writer rank (the in-place all-gather is only safe then), and the result must be the rank-ordered fp32 sum on every replica
    (ParameterAveragingTrainingMaster aggregation, J:325-333, as a sum; the updater divides)."""
    rng = np.random.default_rng(7)
    for world in (2, 3, 4, 8):
        for n in (1, 3, 4, 5, 1023, 1024, 2763841):
            nv = n // 4
            chunk = (nv + world - 1) // world
            owner = np.full(n, -1, np.int64)
            for r in range(world):
                v0 = min(nv, r * chunk); v1 = min(nv, v0 + chunk)
                assert (owner[4 * v0:4 * v1] == -1).all()
                owner[4 * v0:4 * v1] = r
            owner[4 * nv:] = world - 1
            assert (owner >= 0).all() and (owner < world).all(), (world, n)
        n = 1031
        grads = [rng.standard_normal(n).astype(np.float32) for _ in range(world)]
        want = grads[0].copy()
        for r in range(1, world):
            want = (want + grads[r]).astype(np.float32)            # rank order 0..W-1, fp32 at every step: what every replica must hold
        nv = n // 4; chunk = (nv + world - 1) // world
        bufs = [g.copy() for g in grads]
        for r in range(world):                                      # each rank's reduce-scatter + all-gather over its slice (+ the tail on the last rank)
            v0 = min(nv, r * chunk); v1 = min(nv, v0 + chunk)
            idx = np.r_[4 * v0:4 * v1, (np.arange(4 * nv, n) if r == world - 1 else np.arange(0))].astype(np.int64)
            acc = bufs[0][idx].copy()
            for q in range(1, world):
                acc = (acc + bufs[q][idx]).astype(np.float32)
            for q in range(world):
                bufs[q][idx] = acc
        for q in range(world):
            assert np.array_equal(bufs[q], want), (world, q)
