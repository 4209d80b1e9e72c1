"""The structured f32 operand set V on which the FSPT-DM2 binary probes (atan2, pow, min, max and the divisions) are
compared over V x V, GPU against oracle (tests/test_gpu_dm_exhaustive.py) and measured against float64
(tools/dm_accuracy.py).

V holds +-0, every subnormal and normal exponent (a few mantissas each), +-inf, two NaNs, every branch edge of the
model's operation sequences (oracle_math.h / dm_math.cuh) +-2 ulp, and dense runs about the 2^-40 / 2^40 window of the
camera's shared-reciprocal division (device_common.cuh)."""
import numpy as np

# branch edges, as positive magnitudes; V holds each of them +-2 ulp with both signs
EDGES = {
    "atan01 reduction about tan(pi/8)": np.float32(0.4142135679721832),
    "log2 mantissa split": np.float32(1.4142135381698608),
    "smallest normal (log2 subnormal test, div_z's ordinary divisor)": np.float32(1.17549435e-38),
    "largest finite (div_z's ordinary divisor)": np.float32(3.40282347e38),
    "pow's large-x exit": np.float32(3.0e38),
    "sin/cos reduction guard and float->int guard": np.float32(1.0e9),
    "exp2 upper clamp": np.float32(130.0),
    "exp2 lower clamp": np.float32(160.0),
    "exp2 overflow": np.float32(128.0),
    "exp2 last normal": np.float32(126.0),
    "exp2 last subnormal": np.float32(149.0),
    "exp2 underflow": np.float32(150.0),
    # y with y * log2(x) at an exp2 clamp for x = 4, 16 (x = 2, 1/2 give the clamps themselves)
    "pow y reaching 130 at x = 4": np.float32(65.0),
    "pow y reaching 160 at x = 4": np.float32(80.0),
    "pow y reaching 130 at x = 16": np.float32(32.5),
    "pow y reaching 160 at x = 16": np.float32(40.0),
}
# exp2's n = rint(x): arguments that are exact half-integers tie (to even)
EXP2_TIES = [np.float32(v) for v in (0.5, 1.5, 2.5, 3.5, 126.5, 127.5, 128.5, 129.5, 148.5, 149.5, 150.5, 159.5)]
WINDOW = (np.float32(2.0 ** -40), np.float32(2.0 ** 40))  # div3_shared's operand window
WINDOW_RUN = 16  # ulps on each side of each window bound
NANS = (0x7FC00000, 0xFF800001)  # the default quiet NaN and a negative signalling NaN


def reduce_ties(count=12):
    """Positive x for which sin/cos's reduction k = rint(x * 2/pi) ties: the f32 product is exactly m + 1/2."""
    two_over_pi = np.float32(float.fromhex("0x1.45f306p-1"))  # DM_TWO_OVER_PI
    out = []
    for m in range(200):
        x0 = np.float32((m + 0.5) * np.pi / 2)
        xs = (np.arange(-512, 513, dtype=np.int64) + int(x0.view(np.uint32))).astype(np.uint32).view(np.float32)
        hit = xs[(xs * two_over_pi) == np.float32(m + 0.5)]
        if hit.size:
            out.append(hit[0])
        if len(out) == count:
            break
    return out


def _around(v, k):
    b = int(np.float32(v).view(np.uint32))
    return np.arange(b - k, b + k + 1, dtype=np.int64)


def edge_values():
    """Every named edge (EDGES, EXP2_TIES, reduce_ties()) as a positive f32."""
    return list(EDGES.values()) + EXP2_TIES + reduce_ties()


def values(seed=5):
    """V, as f32, sorted by bit pattern, without duplicates."""
    rng = np.random.default_rng(seed)
    mag = [0]
    for lead in range(23):  # subnormals: leading bit `lead`
        lo = 1 << lead
        mag += [lo, lo + 1, 2 * lo - 1, lo + int(rng.integers(0, lo)) if lead else lo]
    for e in range(1, 255):  # normals
        base = e << 23
        mag += [base, base + 1, base + 0x7FFFFF] + [base + int(m) for m in rng.integers(2, 0x7FFFFF, 2)]
    mag.append(0x7F800000)
    for v in edge_values():
        mag += list(_around(v, 2))
    for w in WINDOW:
        mag += list(_around(w, WINDOW_RUN))
    mag = np.array(mag, np.int64)
    mag = mag[mag <= 0x7F800000]  # the largest finite + 2 ulp would be a NaN: the two below are V's NaNs
    bits = np.concatenate([mag, mag | 0x80000000, np.array(NANS, np.int64)]).astype(np.uint32)
    return np.unique(bits).view(np.float32)
