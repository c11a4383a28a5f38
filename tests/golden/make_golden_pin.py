"""Golden fixtures for the distance and quantizer pins of tests/test_oracle_pin.py -- TEST INFRASTRUCTURE.

The inputs are drawn from fixed seeds by the helpers in tests/test_oracle_pin.py; this stores what the UNMODIFIED
REFERENCE (oracle/_ref/libsptag_ref.so through oracle/ref_shim.cpp) returns on them, so that the oracle is checked
against the reference on a machine that does not have it:
  pin/distance_f32.npz        DistanceUtils float variants per SIMD tree (ref_distance_f32_many), first
                              F32_PAIRS_KEPT pairs of every dimension
  pin/distance_int.npz        DistanceUtils int8 / uint8 / int16 through the reference's cpuid dispatch (ref_distance),
                              and the SIMD width that dispatch picked
  pin/quantizer_<case>.npz    the quantizer file the reference was given, and its PQ / OPQ QuantizeVector, SDC L2,
                              ReconstructVector and re-quantisation (RefQuantizer)
The reference sources are not needed to USE the fixtures.  Run (where oracle/_ref exists):  python tests/golden/make_golden_pin.py
"""
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import reflib  # noqa: E402
import test_oracle_pin as pin  # noqa: E402

OUT = os.path.join(HERE, "pin")


def make_f32():
    R = reflib.ref()
    dists = np.empty((2, len(pin.F32_DIMS), len(pin.ISA_WIDTHS), pin.F32_PAIRS_KEPT), np.float32)
    for metric in (0, 1):
        for i, (dim, a, b) in enumerate(pin.f32_distance_inputs()):
            for j, (isa, _) in enumerate(pin.ISA_WIDTHS):
                out = np.empty(pin.F32_PAIRS, np.float32)
                R.ref_distance_f32_many(isa, metric, a.ctypes.data, b.ctypes.data, dim, pin.F32_PAIRS, out.ctypes.data)
                dists[metric, i, j] = out[:pin.F32_PAIRS_KEPT]
    np.savez_compressed(os.path.join(OUT, "distance_f32.npz"), dists=dists)


def make_int():
    R = reflib.ref()
    out = {"width": np.int32({512: 16, 256: 8, 128: 4, 0: 1}[R.ref_isa()])}
    for vt, dt, lo, hi in pin.INT_CASES:
        out[pin.int_case_key(vt, lo, hi)] = np.array(
            [R.ref_distance(metric, vt, a.ctypes.data, b.ctypes.data, dim)
             for metric, dim, a, b in pin.int_distance_inputs(dt, lo, hi)], np.float32)
    np.savez_compressed(os.path.join(OUT, "distance_int.npz"), **out)


def make_quantizer(opq, rtype):
    xs = pin.quantizer_rows(rtype)
    qz = reflib.train_quantizer(xs.astype(np.float32), m=6, ks=256, opq=opq, rtype=rtype, iters=2)
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "q.bin")
        qz.write(path)
        rq = reflib.RefQuantizer(path)
        codes = rq.encode(xs)
        sdc = np.array([rq.l2(codes[i], codes[i + 1]) for i in range(500)], np.float32)
        rec = rq.reconstruct(codes, xs.dtype)
        recoded = rq.encode(rec)
        blob = np.fromfile(path, np.uint8)
    np.savez_compressed(os.path.join(OUT, "quantizer_%s.npz" % pin.quantizer_case_key(opq, rtype)),
                        quantizer_blob=blob, codes=codes[:pin.QUANT_ROWS_KEPT], sdc_l2=sdc,
                        reconstructed=rec[:pin.QUANT_RECON_KEPT], recoded=recoded[:pin.QUANT_ROWS_KEPT])


if __name__ == "__main__":
    if not reflib.have_ref():
        raise SystemExit("oracle/_ref/libsptag_ref.so missing: run `make -C oracle ref` where the reference sources exist")
    os.makedirs(OUT, exist_ok=True)
    make_f32()
    make_int()
    for opq, rtype in pin.QUANTIZER_CASES:
        make_quantizer(opq, rtype)
    for f in sorted(os.listdir(OUT)):
        print("golden pin", f, os.path.getsize(os.path.join(OUT, f)), "bytes")
