"""Helpers shared by the per-element float64 parity tests (tests/test_gpu_aligner_step_parity.py,
tests/test_gpu_t5_objective_parity.py): the GEMM schedule as the library plans it (``td_gemm_schedule``), the tail class of a
GEMM shape, the rows / columns / k-range of its first shared tail tile, and ``Report``, which collects every check's worst
err / tol and prints one JSON line per case."""
import ctypes as C
import json
import time

import torch


def schedule(M, N, K, workers):
    from thinkdiff_mlre_b200 import _lib as L

    f = L.lib().td_gemm_schedule
    n = f(M, N, K, workers, 1, None, 0)
    assert n > 0
    buf = (C.c_int32 * (8 * n))()
    assert f(M, N, K, workers, 1, buf, n) == n
    keys = ("unit", "tile", "kb0", "kb1", "kind", "contrib0", "contrib_n", "range")
    return [dict(zip(keys, buf[8 * i : 8 * i + 8])) for i in range(n)]


def tail_class(M, N, K, workers):
    """"split(c)": a shared tail tile has up to c contributors; "tail unsplit": the last wave is partial but every tile has one
    owner; "no tail": the tiles fill whole waves."""
    owners = [s for s in schedule(M, N, K, workers) if s["kind"] == 1]
    if owners:
        return f"split({max(s['contrib_n'] for s in owners)})"
    tiles = -(-M // 256) * -(-N // 256)
    return "tail unsplit" if tiles % workers else "no tail"


def workers():
    return torch.cuda.get_device_properties(0).multi_processor_count // 2


def shared_tile(M, N, K):
    """Rows, columns and the smallest contributor's k-range [k0, k1) (elements) of the first shared tail tile of the GEMM
    [M, K] x [K, N] on this device."""
    from thinkdiff_mlre_b200 import _lib as L

    segs = schedule(M, N, K, workers())
    owner = next(s for s in segs if s["kind"] == 1)
    c = min((s for s in segs if s["kind"] == 2 and s["tile"] == owner["tile"]), key=lambda s: s["kb1"] - s["kb0"])
    m_blk, n_blk = C.c_int32(-1), C.c_int32(-1)
    # the GEMMs' own tile raster (tile_coords); the row count is rounded up to the multiple of 32 the call checks for, which
    # never changes the number of 256-row blocks
    assert L.lib().td_scatter_tile_owner(owner["tile"], -(-M // 32) * 32, N, 1, -1, C.addressof(m_blk), C.addressof(n_blk)) == 0
    rows = slice(m_blk.value * 256, min(M, m_blk.value * 256 + 256))
    cols = slice(n_blk.value * 256, n_blk.value * 256 + 256)
    return rows, cols, (c["kb0"] * 64, min(K, c["kb1"] * 64))


class Report:
    """Collects every check's worst err / tol and its out-of-bound count, prints one JSON line (prefixed ``tag``), then fails on
    any violation."""

    def __init__(self, label, tag="ALIGNER_STEP_PARITY"):
        self.label, self.tag, self.t0 = label, tag, time.time()
        self.worst, self.bad, self.count, self.info, self.failures = {}, {}, {}, {}, []

    def check(self, name, err, tol):
        ratio = torch.where(tol > 0, err / torch.where(tol > 0, tol, 1.0), torch.where(err > 0, float("inf"), 0.0))
        self.worst[name] = max(self.worst.get(name, 0.0), float(ratio.max()) if ratio.numel() else 0.0)
        self.bad[name] = self.bad.get(name, 0) + int((err > tol).sum())
        self.count[name] = self.count.get(name, 0) + err.numel()
        if bool((err > tol).any()) and name not in self.info.get("first_outside", {}):  # where, for a finding
            i = int(ratio.argmax())
            self.info.setdefault("first_outside", {})[name] = {"index": list(map(int, torch.unravel_index(torch.tensor(i), err.shape))),
                                                               "err": float(err.flatten()[i]), "tol": float(tol.flatten()[i])}

    def require(self, ok, msg):
        if not ok:
            self.failures.append(msg)

    def finish(self):
        fails = [f"{n}: {b} elements outside the bound (worst err/tol {self.worst[n]:.3g})" for n, b in self.bad.items() if b]
        fails += self.failures
        print(self.tag + " " + json.dumps({"case": self.label, "worst_err_over_tol": {k: round(v, 4) for k, v in self.worst.items()},
                                           "elements": self.count, **self.info, "seconds": round(time.time() - self.t0, 1),
                                           "peak_gb": round(torch.cuda.max_memory_allocated() / 2 ** 30, 2)}))
        assert not fails, f"{self.label}: " + "; ".join(fails)
