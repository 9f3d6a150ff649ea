"""Same-process A/B of the top-k step across two library builds (build.py --out=LIB), alternating between them.
Usage: python scripts/ab_rescore.py LIB_A LIB_B [--reps R]

Per shape: the same seeded store and queries go into one store per build; after warm-up, R rounds alternate A and B,
each timing 50 VM_FLAG_ASYNC device-output calls with CUDA events.  One line per shape: the median step time of each
build, B/A, and whether the two builds returned identical lists (one synchronous call each).  The shapes cover the
384-d path neither build changes, stores whose candidate rows need more than three column chunks in shared memory (wide
rows, binary64 stores), small-store dump mode at 1536-d and a store with a near-duplicate cluster at the top."""
import argparse
import ctypes as C
import subprocess

import torch

F32, F64 = 0, 2
ASYNC = 1
CALLS = 50
vp, i64 = C.c_void_p, C.c_int64

# name, rows, dim, store ("f32" | "f64": binary64 rows + fp32 shadow), queries, k, near-duplicate cluster rows
SHAPES = [
    ("1M x 384 fp32", 1_000_000, 384, "f32", 64, 10, 0),
    ("1M x 384 f64", 1_000_000, 384, "f64", 64, 20, 0),
    ("200K x 1536 fp32", 200_000, 1536, "f32", 64, 10, 0),
    ("100K x 1536 f64", 100_000, 1536, "f64", 64, 10, 0),
    ("5000 x 1536 fp32 (dump)", 5_000, 1536, "f32", 30, 10, 0),
    ("100K x 3072 fp32", 100_000, 3072, "f32", 64, 10, 0),
    ("100K x 1536 fp32, 300-row cluster", 100_000, 1536, "f32", 64, 10, 300),
]


class Lib:
    def __init__(self, path):
        self.path = path
        self.L = C.CDLL(path)
        self.L.vm_last_error.restype = C.c_char_p

    def chk(self, rc):
        if rc != 0:
            raise RuntimeError(f"{self.path}: {self.L.vm_last_error().decode()}")

    def store(self, X, kind):
        h = C.c_void_p()
        n, dim = X.shape
        if kind == "f64":
            self.chk(self.L.vm_store_create_exact(C.byref(h), 0, dim, F32, i64(n)))
        else:
            self.chk(self.L.vm_store_create(C.byref(h), 0, dim, F32, i64(n)))
        st = torch.cuda.current_stream().cuda_stream
        self.chk(self.L.vm_store_append(h, vp(X.data_ptr()), F64 if X.dtype == torch.float64 else F32, 1, i64(n), None, vp(st)))
        torch.cuda.synchronize()
        return h

    def topk(self, h, Q, k, out, flags):
        oi, os_, oc = out
        self.chk(self.L.vm_topk(h, vp(Q.data_ptr()), F64 if Q.dtype == torch.float64 else F32, 1, Q.shape[0], k,
                                C.c_double(float("-inf")), 0, 1, flags, vp(oi.data_ptr()), vp(os_.data_ptr()), vp(oc.data_ptr()),
                                1, None, vp(torch.cuda.current_stream().cuda_stream)))


def data(rows, dim, kind, nq, cluster, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    dt = torch.float64 if kind == "f64" else torch.float32
    X = torch.randn((rows, dim), generator=g, device="cuda", dtype=torch.float64)
    Q = torch.randn((nq, dim), generator=g, device="cuda", dtype=torch.float64)
    if cluster:
        centre = torch.randn((dim,), generator=g, device="cuda", dtype=torch.float64)
        X[1000:1000 + cluster] = centre + 1e-7 * torch.randn((cluster, dim), generator=g, device="cuda", dtype=torch.float64)
        Q = centre + 0.05 * torch.randn((nq, dim), generator=g, device="cuda", dtype=torch.float64)
    return X.to(dt), Q.to(dt)


def step_ms(lib, h, Q, k, out):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(CALLS):
        lib.topk(h, Q, k, out, ASYNC)
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / CALLS


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("lib_a")
    ap.add_argument("lib_b")
    ap.add_argument("--reps", type=int, default=7)
    args = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    print("device:", torch.cuda.get_device_name(0), "|", q.stdout.strip())
    libs = [Lib(args.lib_a), Lib(args.lib_b)]
    print(f"A = {args.lib_a}\nB = {args.lib_b}\nmedian step time over {args.reps} alternating rounds of {CALLS} async calls")
    for i, (name, rows, dim, kind, nq, k, cluster) in enumerate(SHAPES):
        X, Q = data(rows, dim, kind, nq, cluster, 100 + i)
        hs = [lib.store(X, kind) for lib in libs]
        del X
        outs = [(torch.empty((nq, k), dtype=torch.int64, device="cuda"), torch.empty((nq, k), dtype=torch.float64, device="cuda"),
                 torch.empty((nq,), dtype=torch.int32, device="cuda")) for _ in libs]
        for lib, h, out in zip(libs, hs, outs):
            lib.topk(h, Q, k, out, 0)
        same = all(torch.equal(a, b) for a, b in zip(*outs))
        for lib, h, out in zip(libs, hs, outs):
            for _ in range(10):
                lib.topk(h, Q, k, out, ASYNC)
        torch.cuda.synchronize()
        t = [[], []]
        for _ in range(args.reps):
            for j in (0, 1):
                t[j].append(step_ms(libs[j], hs[j], Q, k, outs[j]))
        med = [sorted(x)[len(x) // 2] for x in t]
        spread = [f"{min(x):.4f}-{max(x):.4f}" for x in t]
        print(f"{name:36s} k={k:2d} nq={nq:2d}: A {med[0]:.4f} ms [{spread[0]}]  B {med[1]:.4f} ms [{spread[1]}]  "
              f"B/A {med[1] / med[0]:.3f}  identical lists: {same}", flush=True)
        for lib, h in zip(libs, hs):
            lib.chk(lib.L.vm_store_destroy(h))
        del outs
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
