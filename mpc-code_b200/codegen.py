"""Emit straight-line C / CUDA from expression DAGs.

The reference gets its derivative code from CasADi's virtual machine at run time
(``nlpsol`` builds gradient/Jacobian/Hessian functions, ``Control_Calc.py:258``).  Here the
same information is produced once, ahead of time, as source text: one ``static`` function per
map, taking ``const double*`` inputs and ``double*`` outputs, with common sub-expressions shared.
The text compiles unchanged as a CUDA ``__device__`` function (macro ``MPCB_FN``) and as plain C.
"""
from __future__ import annotations

import math
from typing import Dict, List, Sequence, Tuple

from . import symbolic as S
from .sx import SX

_INFIX = {"add": "+", "sub": "-", "mul": "*", "div": "/"}
_CALL1 = {"exp": "MPCB_EXP", "log": "log", "sqrt": "sqrt", "sin": "sin", "cos": "cos", "tan": "tan",
          "tanh": "tanh", "fabs": "fabs", "asin": "asin", "acos": "acos", "atan": "atan",
          "sinh": "sinh", "cosh": "cosh"}
_CMP = {"lt": "<", "le": "<=", "eq": "==", "ne": "!="}


def _lit(v: float) -> str:
    if math.isinf(v):
        return "INFINITY" if v > 0 else "(-INFINITY)"
    if math.isnan(v):
        return "NAN"
    r = repr(float(v))
    return "(%s)" % r if v < 0 else r


class CFunction:
    """One generated function: name, ordered pointer arguments, body text, op statistics."""

    def __init__(self, name: str, inputs: Sequence[Tuple[str, SX]], outputs: Sequence[Tuple[str, SX]],
                 skip_zero_outputs: bool = False, shared_reciprocals: bool = False, cache_in=None):
        self.name = name
        # cache_in = [(argument name, entries), ...]: values of expensive sub-expressions computed by ANOTHER generated
        # function at the same point and handed in through extra ``const double*`` arguments instead of being
        # recomputed (see `expensive_entries`).  entries[i] = ("node", expr) -> arg[i] replaces that node;
        # ("recip", den) -> arg[i] is 1/den and replaces the shared reciprocal of that denominator.
        if cache_in is not None and isinstance(cache_in, tuple):
            cache_in = [cache_in]
        self.cache_in = cache_in
        self.inputs = [(n, v if isinstance(v, SX) else SX(v)) for n, v in inputs]
        self.outputs = [(n, v if isinstance(v, SX) else SX(v)) for n, v in outputs]
        for n, v in self.inputs:
            if not v.is_symbolic():
                raise ValueError("%s: input %s is not purely symbolic" % (name, n))
        self.skip_zero_outputs = skip_zero_outputs
        # a / b is emitted as a * (1 / b) with ONE reciprocal per distinct denominator (and a literal for constant
        # denominators): FP64 division is a ~12-instruction sequence on the GPU, and model right-hand sides and their
        # derivatives divide by the same few quantities many times.  Changes results by at most an ulp per operation.
        self.shared_reciprocals = shared_reciprocals
        self._flat_out = [e for _, o in self.outputs for e in o.elements()]
        self.counts = S.op_counts(self._flat_out)
        self.flops = int(sum(self.counts.values()))

    # -- text ------------------------------------------------------------------
    def signature(self, qualifier="MPCB_FN") -> str:
        args = ["const double* %s" % n for n, _ in self.inputs]
        for cname, _ in (self.cache_in or ()):
            args.append("const double* %s" % cname)
        args += ["double* %s" % n for n, _ in self.outputs]
        return "%s void %s(%s)" % (qualifier, self.name, ", ".join(args))

    def source(self, qualifier="MPCB_FN") -> str:
        ref: Dict[int, str] = {}
        lines: List[str] = []
        known = set()
        for name, var in self.inputs:
            for i, e in enumerate(var.elements()):
                ref[e.uid] = "%s[%d]" % (name, i)
                known.add(e.uid)
        order = S.topo_order(self._flat_out)
        # count uses so that single-use cheap nodes could be inlined; keep it simple: one temp per node
        used_inputs = set()
        recips: Dict[int, str] = {}
        cut_nodes: Dict[int, str] = {}
        if self.cache_in is not None:
            for cname, entries in self.cache_in:
                for i, (kind, e) in enumerate(entries):
                    if kind == "node":
                        cut_nodes[e.uid] = "%s[%d]" % (cname, i)
                    else:
                        recips[e.uid] = "%s[%d]" % (cname, i)
            live = live_nodes(self._flat_out, set(cut_nodes), set(recips) if self.shared_reciprocals else set())
            order = [n for n in order if n.uid in live]
        tcount = 0
        for n in order:
            if n.uid in cut_nodes:
                ref[n.uid] = cut_nodes[n.uid]
                continue
            if n.op == "sym":
                if n.uid not in known:
                    raise ValueError("%s: free symbol %s" % (self.name, n.val))
                used_inputs.add(n.uid)
                continue
            if n.op == "const":
                ref[n.uid] = _lit(n.val)
                continue
            a = [ref.get(c.uid) for c in n.args]        # None only for a denominator hidden behind a cached reciprocal
            op = n.op
            if op == "div" and self.shared_reciprocals:
                den = n.args[1]
                if den.op == "const":
                    rhs = "%s * %s" % (a[0], _lit(1.0 / den.val))
                else:
                    if den.uid not in recips:
                        rname = "r%d" % len(recips)
                        lines.append("  const double %s = MPCB_RCP(%s);" % (rname, a[1]))
                        recips[den.uid] = rname
                    rhs = recips[den.uid] if n.args[0] is S.ONE else "%s * %s" % (a[0], recips[den.uid])
            elif op in _INFIX:
                rhs = "%s %s %s" % (a[0], _INFIX[op], a[1])
            elif op == "neg":
                rhs = "-%s" % a[0]
            elif op == "sq":
                rhs = "%s * %s" % (a[0], a[0])
            elif op in _CALL1:
                rhs = "%s(%s)" % (_CALL1[op], a[0])
            elif op == "sign":
                rhs = "(double)((%s > 0.0) - (%s < 0.0))" % (a[0], a[0])
            elif op == "not":
                rhs = "(%s == 0.0) ? 1.0 : 0.0" % a[0]
            elif op in _CMP:
                rhs = "(%s %s %s) ? 1.0 : 0.0" % (a[0], _CMP[op], a[1])
            elif op == "and":
                rhs = "(%s != 0.0 && %s != 0.0) ? 1.0 : 0.0" % (a[0], a[1])
            elif op == "or":
                rhs = "(%s != 0.0 || %s != 0.0) ? 1.0 : 0.0" % (a[0], a[1])
            elif op == "fmin":
                rhs = "fmin(%s, %s)" % (a[0], a[1])
            elif op == "fmax":
                rhs = "fmax(%s, %s)" % (a[0], a[1])
            elif op == "atan2":
                rhs = "atan2(%s, %s)" % (a[0], a[1])
            elif op == "pow":
                b = n.args[1]
                if b.op == "const" and float(b.val).is_integer() and 0 < abs(b.val) <= 8:
                    k = int(abs(b.val))
                    prod = " * ".join([a[0]] * k)
                    rhs = prod if b.val > 0 else "1.0 / (%s)" % prod
                else:
                    rhs = "pow(%s, %s)" % (a[0], a[1])
            elif op == "if_else":
                rhs = "(%s != 0.0) ? %s : %s" % (a[0], a[1], a[2])
            else:
                raise NotImplementedError(op)
            name = "w%d" % tcount
            tcount += 1
            lines.append("  const double %s = %s;" % (name, rhs))
            ref[n.uid] = name
        for name, var in self.outputs:
            for i, e in enumerate(var.elements()):
                if self.skip_zero_outputs and e is S.ZERO:
                    continue
                lines.append("  %s[%d] = %s;" % (name, i, ref[e.uid]))
        unused = [n for n, v in self.inputs if not any(e.uid in used_inputs for e in v.elements())]
        unused += [cname for cname, _ in (self.cache_in or ())]        # a cache argument may go unused in this function
        unused += [n for n, v in self.outputs if v.numel() == 0]
        head = self.signature(qualifier) + " {"
        voids = ["  (void)%s;" % n for n in unused]
        return "\n".join([head] + voids + lines + ["}"]) + "\n"


BIG_FUNCTION_FLOPS = 3000          # generated functions above this size are not inlined

EXPENSIVE_OPS = frozenset(("exp", "log", "sqrt", "sin", "cos", "tan", "tanh", "asin", "acos", "atan", "sinh", "cosh",
                           "pow", "atan2"))


def live_nodes(roots, cut_nodes, cut_recips):
    """uids reachable from ``roots`` when cached nodes are leaves and cached reciprocals hide their denominators."""
    live, stack = set(), list(roots)
    while stack:
        n = stack.pop()
        if n.uid in live:
            continue
        live.add(n.uid)
        if n.uid in cut_nodes:
            continue
        if n.op == "div" and n.args[1].uid in cut_recips:
            stack.append(n.args[0])
            continue
        stack.extend(n.args)
    return live


def expensive_entries(consumers, tainted, shared_reciprocals=True, recips=True):
    """Expensive sub-expressions (transcendentals, reciprocals of non-constant denominators) of the output lists in
    ``consumers`` that do not depend on the symbols in ``tainted`` - i.e. that a producer evaluated at the same point
    can compute once and pass on.  Entries that end up unused once the others are cut are dropped."""
    roots = [e for c in consumers for e in c]
    order = S.topo_order(roots)
    taint = {e.uid for e in tainted}
    dep: Dict[int, bool] = {}
    for n in order:
        dep[n.uid] = (n.uid in taint) if n.op == "sym" else any(dep[a.uid] for a in n.args)
    entries, seen_den = [], set()
    for n in order:
        if n.op in EXPENSIVE_OPS and not dep[n.uid] and any(a.op != "const" for a in n.args):
            entries.append(("node", n))
        if shared_reciprocals and recips and n.op == "div":
            den = n.args[1]
            if den.op != "const" and not dep[den.uid] and den.uid not in seen_den:
                seen_den.add(den.uid)
                entries.append(("recip", den))
    while True:                                          # drop entries hidden behind other entries
        cut_n = {e.uid for k, e in entries if k == "node"}
        cut_r = {e.uid for k, e in entries if k == "recip"}
        live = live_nodes(roots, cut_n, cut_r)
        used_r = {n.args[1].uid for n in order if n.uid in live and n.op == "div" and n.uid not in cut_n}
        keep = [(k, e) for k, e in entries if (k == "node" and e.uid in live) or (k == "recip" and e.uid in used_r)]
        if len(keep) == len(entries):
            return entries
        entries = keep


def cache_expressions(entries) -> SX:
    """The values a producer must write for `entries` (in order)."""
    return SX([e if k == "node" else S.div(S.ONE, e) for k, e in entries])


def emit_header(guard: str, defines: Dict[str, object], functions: Sequence[CFunction], preamble: str = "") -> str:
    """A self-contained header: size/flag macros followed by the generated functions."""
    out = ["// GENERATED by mpc_code_b200.codegen - do not edit.",
           "#ifndef %s" % guard, "#define %s" % guard,
           "#include <math.h>",
           "#ifndef MPCB_FN",
           "#  ifdef __CUDACC__",
           "#    define MPCB_FN static __host__ __device__ __forceinline__",
           "#  else",
           "#    define MPCB_FN static inline",
           "#  endif",
           "#endif",
           "#ifndef MPCB_FN_BIG",
           "#  ifdef __CUDACC__",
           "#    define MPCB_FN_BIG static __host__ __device__ __noinline__",
           "#  else",
           "#    define MPCB_FN_BIG static __attribute__((noinline))",
           "#  endif",
           "#endif", ""]
    if preamble:
        out.append(preamble)
    out += ["#ifndef MPCB_EXP", "#define MPCB_EXP exp", "#endif", "#ifndef MPCB_RCP", "#define MPCB_RCP(x) (1.0 / (x))", "#endif", ""]
    for k, v in defines.items():
        if isinstance(v, bool):
            v = int(v)
        if isinstance(v, float):
            v = _lit(v)
        out.append("#define %s %s" % (k, v))
    out.append("")
    for f in functions:
        # very large bodies (dense models with many states) are compiled once instead of being inlined into every
        # RK4 stage of every kernel: nvcc's time and the kernels' stack frames grow superlinearly otherwise
        out.append(f.source("MPCB_FN_BIG" if f.flops > BIG_FUNCTION_FLOPS else "MPCB_FN"))
    out.append("#endif")
    return "\n".join(out) + "\n"


# ----------------------------------------------------------------------------
# host-side compilation of generated C (used by tests and by the CPU oracle; the
# product path compiles the same text with nvcc inside the CUDA library instead)
# ----------------------------------------------------------------------------

class CModule:
    """Generated functions compiled with gcc into a shared object and wrapped with ctypes/numpy."""

    def __init__(self, name: str, functions: Sequence[CFunction], build_dir: str, cflags=("-O2",)):
        import ctypes
        import hashlib
        import os
        import subprocess
        import numpy as np
        self._np = np
        self._ct = ctypes
        self.functions = {f.name: f for f in functions}
        src = emit_header("MPCB_GEN_%s_H" % name.upper(), {}, functions,
                          preamble="#undef MPCB_FN\n#define MPCB_FN __attribute__((visibility(\"default\")))\n#undef MPCB_FN_BIG\n#define MPCB_FN_BIG MPCB_FN\n")
        digest = hashlib.sha256((src + " ".join(cflags)).encode()).hexdigest()[:16]
        from .build import build_dir_for
        build_dir = build_dir_for(build_dir, "%s_%s.so" % (name, digest))
        os.makedirs(build_dir, exist_ok=True)
        c_path = os.path.join(build_dir, "%s_%s.c" % (name, digest))
        so_path = os.path.join(build_dir, "%s_%s.so" % (name, digest))
        if not os.path.exists(so_path):
            # several processes may get here at once (the bench's oracle workers): every one compiles its OWN copy of the
            # source and publishes the result by an atomic rename - a shared .c file would be truncated under a running gcc
            tmp_c = "%s.tmp%d.c" % (c_path[:-2], os.getpid())
            tmp_so = so_path + ".tmp%d" % os.getpid()
            with open(tmp_c, "w") as fh:
                fh.write(src)
            try:
                subprocess.run(["gcc", "-shared", "-fPIC", "-std=c99", *cflags, "-o", tmp_so, tmp_c, "-lm"], check=True)
                os.replace(tmp_so, so_path)
            finally:
                if os.path.exists(tmp_c):
                    os.remove(tmp_c)
        self.so_path = so_path
        self._lib = ctypes.CDLL(so_path)
        self._dp = ctypes.POINTER(ctypes.c_double)

    def __getattr__(self, fname):
        if fname.startswith("_") or fname not in self.functions:
            raise AttributeError(fname)
        f = self.functions[fname]
        np, ct = self._np, self._ct
        cfun = getattr(self._lib, fname)
        cfun.restype = None
        in_sizes = [v.numel() for _, v in f.inputs]
        out_shapes = [v.shape for _, v in f.outputs]
        dp = self._dp

        def call(*args):
            if len(args) != len(in_sizes):
                raise TypeError("%s expects %d inputs" % (fname, len(in_sizes)))
            ins = []
            for a, n in zip(args, in_sizes):
                arr = np.ascontiguousarray(np.asarray(a, dtype=np.float64).reshape(-1, order="F"))
                if arr.size != n:
                    raise ValueError("%s: input of size %d, expected %d" % (fname, arr.size, n))
                ins.append(arr)
            outs = [np.zeros(max(s[0] * s[1], 1)) for s in out_shapes]
            cfun(*[a.ctypes.data_as(dp) for a in ins], *[o.ctypes.data_as(dp) for o in outs])
            res = tuple(o[:s[0] * s[1]].reshape(s, order="F") for o, s in zip(outs, out_shapes))
            return res[0] if len(res) == 1 else res
        self.__dict__[fname] = call
        return call
