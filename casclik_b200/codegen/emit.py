"""Scalar DAG -> straight-line CUDA (`__device__ __forceinline__`, fp64) + operation counts.

This is the replacement for CasADi's C code generator + shell JIT on the hot path (SURVEY.md
§2.2): one translation unit per skill that defines `struct Skill` (compile-time sizes, constraint
table, Jacobian sparsity, `eval` / `eval_qp`) and instantiates the hand-written kernels of
csrc/clik_pinv.cuh and csrc/clik_qp.cuh on it.  The same emitter can print plain C (used by the
tests to cross-check the emitted text against the NumPy interpreter with gcc).
"""
import math
import os
import struct

from ..sym import dag
from .lower import KIND_EQ, KIND_SET, KIND_VELEQ

# flops per node for the roofline accounting (SURVEY.md §8d): add/sub/mul/div/sqrt = 1;
# negation, comparisons, selects = 0; transcendental calls are listed separately.
_FLOP_OPS = {"add": 1, "sub": 1, "mul": 1, "div": 1, "sqrt": 1}
_TRANSCENDENTAL = {"sin", "cos", "tan", "asin", "acos", "atan", "atan2", "exp", "log", "pow"}


def literal(v: float) -> str:
    if v != v:
        return "(0.0/0.0)"
    if math.isinf(v):
        return "(1.0/0.0)" if v > 0 else "(-1.0/0.0)"
    if v == int(v) and abs(v) < 1e15:
        return "%d.0" % int(v)
    return float(v).hex()


class Emitter(object):
    """Emits the statements computing a set of nodes, sharing temporaries across calls."""

    def __init__(self, sym_names, const_table=None, sincos_name="sincos", leaves=None):
        self.sym_names = sym_names
        self.name = {}        # node id -> C expression (temp name, symbol name or literal)
        # computed nodes that are inputs of this program (node id -> C lvalue): used as they are, never
        # expanded (the NLP cost functions read the decision-free values eval_nlp_pre hoisted)
        self.leaves = dict(leaves or {})
        self.name.update(self.leaves)
        self.lines = []
        self.counter = 0
        self.hist = {}
        self.const_table = const_table   # list collecting constants that go to the constant bank
        self.sincos_name = sincos_name
        self.sincos_calls = []           # (line index, argument, sin var, cos var)

    def _const(self, v):
        """Constants whose low 32 bits are zero fit an instruction immediate; everything else is
        read from the __constant__ table (a free operand) instead of being built with two moves."""
        if self.const_table is None or v != v or math.isinf(v):
            return literal(v)
        if struct.unpack("<Q", struct.pack("<d", v))[0] & 0xFFFFFFFF == 0:
            return literal(v)
        if v not in self.const_table:
            self.const_table.append(v)
        return "KC[%d]" % self.const_table.index(v)

    def _ref(self, n):
        if n.id in self.leaves:          # (before symbols: a hoisted input row t / q / x / y is a leaf too)
            return self.leaves[n.id]
        if n.op == "const":
            return self._const(n.val)
        if n.op == "sym":
            return self.sym_names[n.id]
        return self.name[n.id]

    def _tmp(self):
        self.counter += 1
        return "v%d" % self.counter

    def require(self, outputs):
        """Make sure every node in `outputs` has been computed."""
        pending = [n for n in outputs if n.op not in ("const", "sym") and n.id not in self.name]
        if not pending:
            return
        order = [n for n in self._topo(pending) if n.op not in ("const", "sym") and n.id not in self.name]
        # pair sin/cos of the same argument into one sincos call
        by_arg = {}
        for n in order:
            if n.op in ("sin", "cos"):
                by_arg.setdefault(n.args[0].id, {})[n.op] = n
        paired = {a: d for a, d in by_arg.items() if len(d) == 2}
        for n in order:
            if n.id in self.name:
                continue
            self.hist[n.op] = self.hist.get(n.op, 0) + 1
            a = [self._ref(x) for x in n.args]
            op = n.op
            if op in ("sin", "cos") and n.args[0].id in paired:
                pair = paired[n.args[0].id]
                s, c = self._tmp(), self._tmp()
                self.lines.append("double %s, %s; %s(%s, &%s, &%s);" % (s, c, self.sincos_name, a[0], s, c))
                if self.sincos_name != "sincos":
                    # deferred range check: patched right after the last fast evaluation
                    self.sincos_calls.append((len(self.lines) - 1, a[0], s, c))
                self.name[pair["sin"].id] = s
                self.name[pair["cos"].id] = c
                other = pair["cos" if op == "sin" else "sin"]
                self.hist[other.op] = self.hist.get(other.op, 0) + 1
                continue
            if op == "add":
                rhs = "%s + %s" % (a[0], a[1])
            elif op == "sub":
                rhs = "%s - %s" % (a[0], a[1])
            elif op == "mul":
                rhs = "%s * %s" % (a[0], a[1])
            elif op == "div":
                rhs = "%s / %s" % (a[0], a[1])
            elif op == "neg":
                rhs = "-%s" % a[0]
            elif op in ("sin", "cos", "tan", "asin", "acos", "atan", "exp", "log", "sqrt", "fabs",
                        "floor", "ceil"):
                rhs = "%s(%s)" % (op, a[0])
            elif op in ("atan2", "pow", "fmin", "fmax"):
                rhs = "%s(%s, %s)" % (op, a[0], a[1])
            elif op == "sign":
                rhs = "(double)((%s > 0.0) - (%s < 0.0))" % (a[0], a[0])
            elif op == "lt":
                rhs = "(%s < %s) ? 1.0 : 0.0" % (a[0], a[1])
            elif op == "le":
                rhs = "(%s <= %s) ? 1.0 : 0.0" % (a[0], a[1])
            elif op == "eq":
                rhs = "(%s == %s) ? 1.0 : 0.0" % (a[0], a[1])
            elif op == "ne":
                rhs = "(%s != %s) ? 1.0 : 0.0" % (a[0], a[1])
            elif op == "and":
                rhs = "(%s != 0.0 && %s != 0.0) ? 1.0 : 0.0" % (a[0], a[1])
            elif op == "or":
                rhs = "(%s != 0.0 || %s != 0.0) ? 1.0 : 0.0" % (a[0], a[1])
            elif op == "not":
                rhs = "(%s == 0.0) ? 1.0 : 0.0" % a[0]
            elif op == "if_else":
                rhs = "(%s != 0.0) ? %s : %s" % (a[0], a[1], a[2])
            else:  # pragma: no cover
                raise NotImplementedError(op)
            t = self._tmp()
            self.lines.append("const double %s = %s;" % (t, rhs))
            self.name[n.id] = t

    def _topo(self, outputs):
        if not self.leaves:
            return dag.topo(outputs)
        seen, stack = {}, list(outputs)
        while stack:
            n = stack.pop()
            if n.id in seen:
                continue
            seen[n.id] = n
            if n.id not in self.leaves:
                stack.extend(n.args)
        return [seen[k] for k in sorted(seen)]

    def assign(self, lhs, node):
        self.require([node])
        self.roots = getattr(self, "roots", [])
        self.roots.append(node)
        self.lines.append("%s = %s;" % (lhs, self._ref(node)))

    def finish(self):
        """Emitted statements, with the out-of-range fix-up of the branch-free sincos calls: every
        run of fast calls whose arguments are available is followed by ONE combined range test,
        so the compiler is free to interleave the polynomial chains of all joints."""
        if not self.sincos_calls:
            return list(self.lines)
        # group calls whose arguments are inputs/early values: a call can join the current group
        # only if its argument does not depend on a sin/cos result of the same group; kinematic
        # chains take sin/cos of the raw joint angles, so in practice there is one group.
        out = list(self.lines)
        groups, cur, produced = [], [], set()
        for idx, arg, sv, cv in self.sincos_calls:
            if cur and any(p in self._deps_text(arg) for p in produced):
                groups.append(cur)
                cur, produced = [], set()
            cur.append((idx, arg, sv, cv))
            produced.update((sv, cv))
        groups.append(cur)
        import re
        def_line = {}
        for i, ln in enumerate(self.lines):
            if ln.startswith("const double "):
                def_line[ln[len("const double "):].split(" = ", 1)[0]] = i
        for g in reversed(groups):
            first = g[0][0]
            # lines to hoist to the position of the group's first call: the calls themselves and
            # every definition after `first` that one of their arguments depends on
            hoist = set(idx for idx, _, _, _ in g)
            for _, arg, _, _ in g:
                for name in self._deps_text(arg):
                    i = def_line.get(name)
                    if i is not None and i > first:
                        hoist.add(i)
            last = g[-1][0]
            region = list(range(first, last + 1))
            moved = [out[i] for i in region if i in hoist]
            rest = [out[i] for i in region if i not in hoist]
            test = " && ".join("clik::sincos_in_range(%s)" % arg for _, arg, _, _ in g)
            fix = ["if (!(%s)) {" % test]
            for _, arg, sv, cv in g:
                fix.append("  if (!clik::sincos_in_range(%s)) { const clik::SinCos sc_ = clik::sincos_slow(%s); %s = sc_.s; %s = sc_.c; }"
                           % (arg, arg, sv, cv))
            fix.append("}")
            out[first:last + 1] = moved + fix + rest
        return out

    def _deps_text(self, arg):
        # arguments are temporaries or symbols; a conservative textual dependency walk
        seen, stack = set(), [arg]
        defs = getattr(self, "_defs", None)
        if defs is None:
            defs = {}
            for ln in self.lines:
                if ln.startswith("const double "):
                    name, rhs = ln[len("const double "):].split(" = ", 1)
                    defs[name] = rhs
            self._defs = defs
        while stack:
            a = stack.pop()
            if a in seen:
                continue
            seen.add(a)
            rhs = defs.get(a)
            if rhs:
                import re
                stack.extend(re.findall(r"v\d+", rhs))
        return seen

    def read_masks(self, syms):
        """(t, q, x, y) bit masks of the input rows the emitted program reads."""
        ids = {n.id for n in dag.symbols_of(getattr(self, "roots", []))}
        def mask(nodes):
            return sum(1 << j for j, n in enumerate(nodes) if n.id in ids and j < 32) | \
                (0xffffffff ^ ((1 << min(len(nodes), 32)) - 1) if len(nodes) > 32 else 0)
        return (1 if syms.t[0].id in ids else 0, mask(syms.q), mask(syms.x), mask(syms.y))

    def inputs_read(self):
        """Number of distinct input scalars (t, q_i, x_i, y_i) the emitted program reads: loads of
        unused inputs are dead code in the kernel, so only these count as algorithmic traffic."""
        return len(dag.symbols_of(getattr(self, "roots", [])))

    def counts(self):
        flops = sum(_FLOP_OPS.get(op, 0) * k for op, k in self.hist.items())
        trans = {op: k for op, k in self.hist.items() if op in _TRANSCENDENTAL}
        return {"flops": flops, "transcendentals": trans, "ops": dict(self.hist)}


# ----------------------------------------------------------------------------------------------
# hand-written-kernel flop model (mode 0 of the static path), mirrors csrc/clik_pinv.cuh
# ----------------------------------------------------------------------------------------------

def _chol_flops(k):
    f = 0
    for j in range(k):
        f += 2 * j + 2                      # diagonal fma chain + rsqrt (sqrt + div)
        f += (k - j - 1) * (2 * j + 1)      # column below the diagonal
    return f


def _subst_flops(k):
    return 2 * sum(2 * i + 1 for i in range(k))   # forward + backward substitution


def _spd_solve_flops(k):
    return _chol_flops(k) + _subst_flops(k)


def pinv_mode0_flops(prog):
    """Arithmetic of the accepted-mode-0 path in clik_pinv.cuh for this skill (fma = 2)."""
    ns = prog.ns
    nz = {}
    for b in prog.blocks:
        for r in range(b["rows"]):
            nz[b["row0"] + r] = [n is not dag.ZERO for n in b["J"][r]]

    def dot_rows(ra, rb):
        c = sum(1 for j in range(ns) if nz[ra][j] and nz[rb][j])
        return max(2 * c - 1, 0)

    def pinv_times(rows):
        k = len(rows)
        wide = (ns >= k) if prog.damped else (k < ns)
        f = 0
        if wide:
            for a in range(k):
                for c in range(a + 1):
                    f += dot_rows(rows[a], rows[c]) + (1 if a == c else 0)
            f += _spd_solve_flops(k)
            for j in range(ns):
                f += max(2 * sum(1 for a in rows if nz[a][j]) - 1, 0)
        else:
            for i in range(ns):
                for c in range(i + 1):
                    f += max(2 * sum(1 for a in rows if nz[a][i] and nz[a][c]) - 1, 0) + (1 if i == c else 0)
            for j in range(ns):
                f += max(2 * sum(1 for a in rows if nz[a][j]) - 1, 0)
            f += _spd_solve_flops(ns)
        return f

    def nullspace(rows):
        f = sum(max(2 * sum(nz[a]) - 1, 0) for a in rows)
        return f + pinv_times(rows) + ns

    flops = 0
    stack = []
    for b in prog.blocks:
        own = list(range(b["row0"], b["row0"] + b["rows"]))
        if b["kind"] in (KIND_EQ, KIND_VELEQ):
            flops += pinv_times(own)
            if not stack:
                flops += ns
                stack = stack + own
                if b["kind"] == KIND_EQ:
                    if getattr(prog, "fuse_first_eq", True):
                        # first_equality_twice: one more substitution on the same factor
                        k = len(own)
                        wide = (ns >= k) if prog.damped else (k < ns)
                        flops += (_subst_flops(k) + 2 * k) if wide else (_subst_flops(ns) + 2 * ns)
                        flops -= ns          # a single v += w
                    else:
                        flops += nullspace(stack) + ns
                    stack = stack + own
            else:
                flops += nullspace(stack) + ns
                stack = stack + own
        elif b["kind"] == KIND_SET:
            flops += 2 * sum(nz[b["row0"]]) + 4     # in-tangent-cone test of the inactive set
    return flops


# ----------------------------------------------------------------------------------------------
# translation unit
# ----------------------------------------------------------------------------------------------

def _switch(name, values, ret="int"):
    body = " ".join("case %d: return %s;" % (i, v) for i, v in enumerate(values))
    return ("  __host__ __device__ static constexpr %s %s(int c) { switch (c) { %s default: return 0; } }"
            % (ret, name, body))


def emit_skill(pinv=None, qp=None, label="skill", block_threads=None, min_blocks=None, qp_fast_min_blocks=None,
               nlp=None, nlp_tol=1e-10, vjp=False):
    """-> (source text, meta dict).  `pinv`: PinvProgram or None, `qp`: QpProgram or None; or `nlp`:
    NlpProgram (an NLP-only image, stopping tolerance `nlp_tol`).  `vjp`: also append the reverse-mode
    derivative kernel of the QP / NLP step (clik_vjp.cuh) after the multiplier kernel, for skills that have
    one; everything emitted before it is the same text as with vjp=False.
    Tuning knobs (also settable through the environment for experiments): CLIK_BLOCK,
    CLIK_MINBLOCKS, CLIK_CONSTBANK (1), CLIK_FAST_SINCOS (1)."""
    if block_threads is None:
        block_threads = int(os.environ.get("CLIK_BLOCK", "128"))
    if nlp is not None:
        if pinv is not None or qp is not None:
            raise ValueError("an NLP image holds the NLP kernels only")
        return _emit_nlp(nlp, label, block_threads, nlp_tol, vjp)
    env_min_blocks = int(os.environ.get("CLIK_MINBLOCKS", "0"))
    if min_blocks is None:
        min_blocks = env_min_blocks
    const_table = [] if os.environ.get("CLIK_CONSTBANK", "1") == "1" else None
    sincos_name = "clik::sincos_fast" if os.environ.get("CLIK_FAST_SINCOS", "1") == "1" else "sincos"
    ref = pinv if pinv is not None else qp
    if ref is None:
        raise ValueError("nothing to emit")
    nq, nxv, ny = ref.n_rob, ref.n_virt, ref.n_in
    meta = {"label": label, "n_robot": nq, "n_virtual": nxv, "n_input": ny,
            "has_pinv": pinv is not None, "has_qp": qp is not None,
            "n_modes": 1, "qp_n": 0, "qp_m": 0, "block_threads": block_threads}
    out = []
    out.append("// generated by casclik_b200.codegen for skill %r -- do not edit" % label)
    out.append('#include "clik_math.cuh"')
    out.append('#include "clik_pinv.cuh"')
    out.append('#include "clik_pinv_group.cuh"')
    out.append('#include "clik_qp.cuh"')
    out.append("")
    pre_struct = []
    struct_at = len(out)
    out.append("struct Skill {")
    out.append("  static constexpr int NQ = %d, NX = %d, NY = %d, NS = %d;" % (nq, nxv, ny, nq + nxv))
    out.append("  static constexpr int BLOCK = %d;   // threads per CTA of the step kernels" % block_threads)
    sig = ("const double t, const double (&q)[%d], const double (&x)[%d], const double (&y)[%d]"
           % (max(nq, 1), max(nxv, 1), max(ny, 1)))

    if pinv is not None:
        from ..controllers._modes import activation_map
        amap = activation_map(pinv.n_sets)
        masks = [sum(b << k for k, b in enumerate(row)) for row in amap] or [0]
        meta["n_modes"] = len(masks)
        kinds = [b["kind"] for b in pinv.blocks]
        out.append("  static constexpr int NC = %d, M = %d, NSETS = %d, NMODES = %d, MAXROWS = %d;"
                   % (len(pinv.blocks), pinv.m, pinv.n_sets, len(masks), pinv.max_rows))
        out.append("  static constexpr bool DAMPED = %s;" % ("true" if pinv.damped else "false"))
        out.append("  static constexpr double LAMBDA = %s;" % literal(pinv.damping))
        fuse = os.environ.get("CLIK_FUSE_FIRST_EQ", "1") == "1"
        pinv.fuse_first_eq = fuse
        out.append("  static constexpr bool FUSE_FIRST_EQ = %s;" % ("true" if fuse else "false"))
        meta["fuse_first_eq"] = fuse
        out.append(_switch("kind", kinds))
        out.append(_switch("row0", [b["row0"] for b in pinv.blocks]))
        out.append(_switch("rows", [b["rows"] for b in pinv.blocks]))
        out.append(_switch("set_index", [max(b["set_index"], 0) for b in pinv.blocks]))
        out.append("  static constexpr bool MULTIDIM = %s;   // options[\"multidim_sets\"]" % ("true" if pinv.multidim else "false"))
        row_is_set = []
        for b in pinv.blocks:
            row_is_set += [1 if b["kind"] == KIND_SET else 0] * b["rows"]
        out.append(_switch("row_is_set", row_is_set, ret="bool"))
        out.append("  static constexpr bool CONV_LAST = %s;   // options[\"converge_final_set_to_max\"] applies"
                   % ("true" if pinv.conv_last else "false"))
        eq_slots, nxt = [], 0
        for bi, b in enumerate(pinv.blocks):
            if b["kind"] in (KIND_EQ, KIND_VELEQ) or (pinv.conv_last and bi == len(pinv.blocks) - 1):
                eq_slots.append(nxt)
                nxt += 1
            else:
                eq_slots.append(0)
        out.append("  static constexpr int NEQC = %d;   // Eq / VelEq constraints" % nxt)
        out.append(_switch("eq_index", eq_slots))
        rowmask = []
        for b in pinv.blocks:
            for r in range(b["rows"]):
                rowmask.append(sum((1 << j) for j, n in enumerate(b["J"][r]) if n is not dag.ZERO))
        if pinv.ns > 63:
            raise NotImplementedError("more than 63 state variables")
        out.append("  __host__ __device__ static constexpr bool jnz(int r, int j) {")
        out.append("    constexpr unsigned long long m[%d] = {%s};" % (
            len(rowmask), ", ".join("0x%xULL" % v for v in rowmask)))
        out.append("    return (m[r] >> j) & 1ULL;")
        out.append("  }")
        if len(masks) > 4096:
            raise NotImplementedError("more than 12 SetConstraints (4096 modes)")
        pre_struct.append("__device__ const unsigned short clik_mode_tab[%d] = {%s};" % (
            len(masks), ", ".join(str(v) for v in masks)))
        out.append("  __device__ static __forceinline__ unsigned mode_mask(int mi) { return clik_mode_tab[mi]; }")
        inv = [0] * len(masks)
        for mi, mk in enumerate(masks):
            inv[mk] = mi
        pre_struct.append("__device__ const unsigned short clik_mode_inv[%d] = {%s};   // mask -> mode index" % (
            len(masks), ", ".join(str(v) for v in inv)))
        out.append("  __device__ static __forceinline__ unsigned mode_index(unsigned mask) { return clik_mode_inv[mask]; }")
        # modes compiled on the static register path: all of them when there are at most 8,
        # otherwise those with at most two active sets if that is at most 64 modes (iiwa: 29 of
        # 128, which covers 99.6 % of the random instances of configs[2]), else mode 0 + singles
        ns_ = pinv.n_sets
        upto2 = 1 + ns_ + ns_ * (ns_ - 1) // 2
        default_static = len(masks) if len(masks) <= 8 else (upto2 if upto2 <= 64 else 1 + ns_)
        unit_sets = pinv.unit_sets if os.environ.get("CLIK_UNIT_SETS", "1") == "1" else None
        meta["pinv_unit_sets"] = bool(unit_sets)
        out.append("  static constexpr bool UNIT_SETS = %s;   // every set bounds one coordinate: closed-form modes"
                   % ("true" if unit_sets else "false"))
        out.append(_switch("set_unit_col", [c for c, _ in (unit_sets or [(0, 1.0)])]))
        out.append(_switch("set_unit_coef", [literal(k) for _, k in (unit_sets or [(0, 1.0)])], ret="double"))
        if unit_sets:
            default_static = 1
        n_static = int(os.environ.get("CLIK_NSTATIC", "0")) or default_static
        n_static = max(1, min(n_static, len(masks)))
        meta["pinv_static_modes"] = n_static
        # skills with a run-time tail of the activation map: fast pass (static modes) + group pass
        has_tail = (not unit_sets) and n_static < len(masks)
        meta["pinv_split"] = has_tail and os.environ.get("CLIK_PINV_SPLIT", "1") == "1"
        meta["pinv_group"] = meta["pinv_split"] or os.environ.get("CLIK_PINV_GROUP", "0") == "1"
        out.append("  static constexpr int NSTATIC = %d;   // leading modes instantiated on the static path" % n_static)
        out.append(_switch("static_mask", masks[:n_static], ret="unsigned"))
        em = Emitter(pinv.syms.names, const_table, sincos_name)
        body = []
        for b in pinv.blocks:
            for r in range(b["rows"]):
                gr = b["row0"] + r
                for j in range(pinv.ns):
                    em.assign("d.J[%d]" % (gr * pinv.ns + j), b["J"][r][j])
                if b["kind"] in (KIND_EQ, KIND_VELEQ):
                    em.assign("d.des[%d]" % gr, b["des"][r])
                elif b["kind"] == KIND_SET:
                    if "des" in b:      # final set with converge_final_set_to_max
                        em.assign("d.des[%d]" % gr, b["des"][r])
                    em.assign("d.e[%d]" % gr, b["e"][r])
                    em.assign("d.jt[%d]" % gr, b["jt"][r])
                    em.assign("d.smin[%d]" % gr, b["smin"][r])
                    em.assign("d.smax[%d]" % gr, b["smax"][r])
                    if pinv.multidim:
                        em.assign("d.rmask[%d]" % gr, b["rmask"][r])
        body = em.finish()
        out.append("  __device__ static __forceinline__ void eval(%s, clik::PinvData<Skill>& d) {" % sig)
        out += ["    " + ln for ln in body]
        out.append("  }")
        # rows staged through shared memory by the TMA driver: only the inputs the program reads
        read_ids = {n.id for n in dag.symbols_of(em.roots)}
        staged = []          # (array name, row, C lvalue)
        if pinv.syms.t[0].id in read_ids:
            staged.append(("t", 0, "tv"))
        for arr, nodes, lv in (("q", pinv.syms.q, "qv"), ("x", pinv.syms.x, "xv"), ("y", pinv.syms.y, "yv")):
            for j, n in enumerate(nodes):
                if n.id in read_ids:
                    staged.append((arr, j, "%s[%d]" % (lv, j)))
        t_staged = bool(staged) and staged[0][0] == "t"
        out.append("  static constexpr int NIN = %d;   // input rows read by eval (t first if read)" % len(staged))
        out.append("  static constexpr bool T_STAGED = %s;" % ("true" if t_staged else "false"))
        out.append("  __device__ static __forceinline__ const double* in_row(int k, long long N, const double* t,")
        out.append("      const double* q, const double* x, const double* y) {")
        out.append("    switch (k) {")
        for k, (arr, j, _) in enumerate(staged):
            out.append("      case %d: return %s + %dLL * N;" % (k, arr, j) if arr != "t" else
                       "      case %d: return t;" % k)
        out.append("      default: return q;")
        out.append("    }")
        out.append("  }")
        out.append("  template <int TILE> __device__ static __forceinline__ void unstage(const double (*b)[TILE], int tid,")
        out.append("      int t_stride, double& tv, double (&qv)[%d], double (&xv)[%d], double (&yv)[%d]) {"
                   % (max(nq, 1), max(nxv, 1), max(ny, 1)))
        for k, (arr, j, lv) in enumerate(staged):
            if arr == "t":
                out.append("    if (t_stride != 0) tv = b[%d][tid];" % k)
            else:
                out.append("    %s = b[%d][tid];" % (lv, k))
        out.append("  }")
        meta["pinv_read_masks"] = em.read_masks(pinv.syms)
        meta["pinv_staged_rows"] = len(staged)
        meta["pinv_t_read"] = t_staged
        cnt = em.counts()
        meta["pinv_eval"] = cnt
        meta["pinv_algebra_flops_mode0"] = pinv_mode0_flops(pinv)
        meta["pinv_flops_mode0"] = cnt["flops"] + meta["pinv_algebra_flops_mode0"]
        meta["pinv_inputs_read"] = em.inputs_read()
        meta["pinv_bytes_per_step"] = 8 * em.inputs_read() + 8 * (nq + nxv) + 4
        meta["jacobian_nnz"] = sum(bin(v).count("1") for v in rowmask)
        meta["rows"] = pinv.m

    if qp is not None:
        meta["qp_n"], meta["qp_m"] = qp.nx, qp.m
        out.append("  static constexpr int QN = %d, QM = %d;" % (qp.nx, qp.m))
        md, mu = len(qp.dense_rows), len(qp.unit_rows)
        env = os.environ.get("CLIK_QP_STRUCT")
        qstruct = (md <= 6 and qp.nx <= 12 and qp.m <= 32) if env is None else (env == "1")
        meta["qp_structured"] = qstruct
        meta["qp_dense_rows"], meta["qp_unit_rows"] = md, mu
        out.append("  static constexpr bool QSTRUCT = %s;   // register-resident structured solver" %
                   ("true" if qstruct else "false"))
        em = Emitter(qp.syms.names, const_table, sincos_name)
        if qstruct:
            out.append("  static constexpr int QMD = %d, QMU = %d;   // dense rows, single-variable rows" % (md, mu))
            out.append("  static constexpr bool QP_CRASH = %s;   // closed-form working-set guess for cold solves" %
                       ("true" if os.environ.get("CLIK_QP_CRASH", "1") == "1" else "false"))
            out.append("  static constexpr bool QP_CRASH_FINAL = %s;   // a certified prediction is returned as is" %
                       ("true" if os.environ.get("CLIK_QP_CRASH_FINAL", "1") == "1" else "false"))
            crash_final = os.environ.get("CLIK_QP_CRASH_FINAL", "1") == "1" and os.environ.get("CLIK_QP_CRASH", "1") == "1"
            meta["qp_split"] = crash_final and os.environ.get("CLIK_QP_SPLIT", "1") == "1"
            out.append("  static constexpr bool QP_CRASH_SINGLE = %s;   // one-row-per-pass prediction passes before the iteration" %
                       ("true" if os.environ.get("CLIK_QP_CRASH_SINGLE", "1") == "1" else "false"))
            out.append("  static constexpr int QP_FAST_PASSES = %d;   // prediction passes in the fast launch (the tail continues)" %
                       int(os.environ.get("CLIK_QP_FAST_PASSES", "3")))
            out.append("  static constexpr int QP_FLIP_PASSES = %d;   // first passes in which a released variable may go straight to another bound" %
                       int(os.environ.get("CLIK_QP_FLIP_PASSES", "2")))
            out.append("  static constexpr bool QP_EQ_START = %s;" %
                       ("true" if os.environ.get("CLIK_QP_EQ_START", "0") == "1" else "false"))
            # structural zeros of the dense rows (slack columns of other rows, joints a task does not depend on):
            # skipped at compile time in the prediction passes, like jnz() in the pinv algebra
            admask = [sum((1 << j) for j in range(qp.nx) if qp.A[r][j] is not dag.ZERO) for r in qp.dense_rows] or [0]
            if os.environ.get("CLIK_QP_ADNZ", "1") != "1":
                admask = [(1 << qp.nx) - 1 for _ in admask]
            meta["qp_dense_nnz"] = sum(bin(v).count("1") for v in admask)
            out.append("  __host__ __device__ static constexpr bool ad_nz(int a, int j) {")
            out.append("    constexpr unsigned m[%d] = {%s};" % (len(admask), ", ".join("0x%xu" % v for v in admask)))
            out.append("    return (m[a] >> j) & 1u;")
            out.append("  }")
            out.append(_switch("dense_row", qp.dense_rows or [0]))
            out.append(_switch("unit_row", [r for r, _, _ in qp.unit_rows] or [0]))
            out.append(_switch("unit_col", [c for _, c, _ in qp.unit_rows] or [0]))
            out.append(_switch("unit_coef", [literal(k) for _, _, k in qp.unit_rows] or ["1.0"], ret="double"))
            for a, r in enumerate(qp.dense_rows):
                for j in range(qp.nx):
                    em.assign("d.Ad[%d]" % (a * qp.nx + j), qp.A[r][j])
                em.assign("d.lbd[%d]" % a, qp.lb[r])
                em.assign("d.ubd[%d]" % a, qp.ub[r])
            for i, (r, _, _) in enumerate(qp.unit_rows):
                em.assign("d.lbu[%d]" % i, qp.lb[r])
                em.assign("d.ubu[%d]" % i, qp.ub[r])
            for j in range(qp.nx):
                em.assign("d.s[%d]" % j, dag.div(dag.ONE, dag.sqrt(qp.h[j])))
            out.append("  __device__ static __forceinline__ void eval_qps(%s, clik::QpSData<Skill>& d) {" % sig)
        else:
            for r in range(qp.m):
                for j in range(qp.nx):
                    em.assign("d.A[%d]" % (r * qp.nx + j), qp.A[r][j])
                em.assign("d.lb[%d]" % r, qp.lb[r])
                em.assign("d.ub[%d]" % r, qp.ub[r])
            for j in range(qp.nx):
                em.assign("d.h[%d]" % j, qp.h[j])
            out.append("  __device__ static __forceinline__ void eval_qp(%s, clik::QpData<Skill>& d) {" % sig)
        out += ["    " + ln for ln in em.finish()]
        out.append("  }")
        meta["qp_eval"] = em.counts()
        meta["qp_read_masks"] = em.read_masks(qp.syms)
        # rows the program reads: only those are fetched and checked for NaN / inf (the host entry
        # points upload only those, the others are undefined in the device copy)
        out.append("  static constexpr unsigned QP_READ_T = %du, QP_READ_Q = 0x%xu, QP_READ_X = 0x%xu, QP_READ_Y = 0x%xu;"
                   % meta["qp_read_masks"])
        meta["qp_inputs_read"] = em.inputs_read()
        meta["qp_bytes_per_step"] = 8 * em.inputs_read() + 8 * qp.nx + 4 + 8

    out.append("};")
    out.append("")
    if const_table:
        pre_struct.append("__constant__ double KC[%d] = {%s};" % (
            len(const_table), ", ".join(literal(v) for v in const_table)))
    out[struct_at:struct_at] = pre_struct
    bounds = "__launch_bounds__(%d%s)" % (block_threads, (", %d" % min_blocks) if min_blocks else "")
    if pinv is not None:
        out.append('extern "C" __global__ void %s clik_pinv_kernel(' % bounds)
        out.append("    long long N, long long ld, const double* t, int t_stride, const double* q, const double* x,")
        out.append("    const double* y, double* qdot, double* xdot, int* mode) {")
        unroll = int(os.environ.get("CLIK_UNROLL", "1"))
        meta["pinv_unroll"] = unroll
        pf = int(os.environ.get("CLIK_PREFETCH_CTAS", "0"))
        meta["pinv_prefetch_ctas"] = pf
        out.append("  clik::pdl_launch_dependents();")
        out.append("  clik::pinv_step<Skill, %d, %d>(N, ld, t, t_stride, q, x, y, qdot, xdot, mode);" % (unroll, pf))
        out.append("  clik::pdl_wait();")
        out.append("}")
        # (the rollout kernel keeps its state across steps in registers: the step kernel's occupancy cap,
        # chosen from the step kernel's spill size, does not transfer to it)
        rbounds = "__launch_bounds__(%d%s)" % (block_threads, (", %d" % env_min_blocks) if env_min_blocks else "")
        out.append('extern "C" __global__ void %s clik_pinv_rollout_kernel(' % rbounds)
        out.append("    long long N, long long ld, int steps, double dt, const double* t0, int t_stride, double* q, double* x,")
        out.append("    const double* y, double vmax_q, double vmax_x, double* qdot_last, double* xdot_last,")
        out.append("    int* mode_last, int* n_failed) {")
        out.append("  clik::pinv_rollout<Skill>(N, ld, steps, dt, t0, t_stride, q, x, y, vmax_q, vmax_x, qdot_last,")
        out.append("                            xdot_last, mode_last, n_failed);")
        out.append("}")
        if meta.get("pinv_split"):
            out.append('extern "C" __global__ void %s clik_pinv_fast_kernel(' % bounds)
            out.append("    long long N, long long ld, const double* t, int t_stride, const double* q, const double* x,")
            out.append("    const double* y, double* qdot, double* xdot, int* mode) {")
            out.append("  clik::pdl_launch_dependents();")
            out.append("  clik::pinv_step<Skill, %d, %d, true>(N, ld, t, t_stride, q, x, y, qdot, xdot, mode);" % (unroll, pf))
            out.append("  clik::pdl_wait();")
            out.append("}")
        if meta.get("pinv_group"):
            # sub-warp mapping (clik_pinv_group.cuh): tail of the fast pass, or whole batches on request
            out.append('extern "C" __global__ void __launch_bounds__(clik::GroupGeometry<Skill>::BLOCK) clik_pinv_group_kernel(')
            out.append("    long long N, long long ld, const double* t, int t_stride, const double* q, const double* x,")
            out.append("    const double* y, double* qdot, double* xdot, int* mode, int from_mode, int only_pending) {")
            out.append("  clik::pdl_launch_dependents();")
            out.append("  clik::pdl_wait();   // reads the mode[] the fast pass wrote")
            out.append("  clik::pinv_group_step<Skill>(N, ld, t, t_stride, q, x, y, qdot, xdot, mode, from_mode, only_pending);")
            out.append("}")
        # TMA-staged persistent variant (DESIGN.md §4.1 / §4.2b): slower than the plain kernel when launches run
        # one after the other, faster for HBM-leaning skills when batches alternate over two streams.  Emitted for
        # small single-launch skills, used on request (clik_skill_set_staging); CLIK_TMA=1 emits and uses it, 0 never.
        tma_env = os.environ.get("CLIK_TMA")
        emit_tma = tma_env == "1" or (tma_env is None and not meta.get("pinv_split")
                                      and 0 < meta.get("pinv_staged_rows", 0) <= 16 and pinv.m <= 8)
        meta["pinv_staged_kernel"] = bool(emit_tma)
        if emit_tma:
            out.append("#ifndef CLIK_NO_TMA_KERNEL   // (the host test harness cannot compile the mbarrier / bulk-copy PTX)")
            out.append('extern "C" __global__ void %s clik_pinv_tma_kernel(' % bounds)
            out.append("    long long N, long long ld, const double* t, int t_stride, const double* q, const double* x,")
            out.append("    const double* y, double* qdot, double* xdot, int* mode) {")
            out.append("  clik::pdl_launch_dependents();")
            out.append("  clik::pinv_step_tma<Skill, %d, %d>(N, ld, t, t_stride, q, x, y, qdot, xdot, mode);"
                       % (block_threads, int(os.environ.get("CLIK_STAGES", "2"))))
            out.append("  clik::pdl_wait();")
            out.append("}")
            out.append("#endif")
    if qp is not None:
        qmin = int(os.environ.get("CLIK_QP_MINBLOCKS", "0"))
        qbounds = "__launch_bounds__(%d%s)" % (block_threads, (", %d" % qmin) if qmin else "")
        out.append('extern "C" __global__ void %s clik_qp_kernel(' % qbounds)
        out.append("    long long N, long long ld, const double* t, int t_stride, const double* q, const double* x,")
        out.append("    const double* y, const double* x0, const unsigned* active0, double* sol, int* status,")
        out.append("    unsigned* active, int max_iter) {")
        out.append("  clik::pdl_launch_dependents();")
        out.append("  clik::qp_step<Skill, clik::QP_FULL>(N, ld, t, t_stride, q, x, y, x0, active0, sol, status, active, max_iter);")
        out.append("  clik::pdl_wait();")
        out.append("}")
        if meta.get("qp_split"):
            # fast pass (working-set prediction only) + tail pass (full solver on what it left pending)
            fmin = qp_fast_min_blocks if qp_fast_min_blocks is not None else int(os.environ.get("CLIK_QP_FAST_MINBLOCKS", "0"))
            meta["qp_fast_min_blocks"] = fmin
            out.append('extern "C" __global__ void __launch_bounds__(%d%s) clik_qp_fast_kernel(' % (
                block_threads, (", %d" % fmin) if fmin else ""))
            out.append("    long long N, long long ld, const double* t, int t_stride, const double* q, const double* x,")
            out.append("    const double* y, const double* x0, const unsigned* active0, double* sol, int* status,")
            out.append("    unsigned* active, int max_iter) {")
            out.append("  clik::pdl_launch_dependents();")
            out.append("  clik::qp_step<Skill, clik::QP_FAST>(N, ld, t, t_stride, q, x, y, x0, active0, sol, status, active, max_iter);")
            out.append("  clik::pdl_wait();")
            out.append("}")
            out.append('extern "C" __global__ void %s clik_qp_tail_kernel(' % qbounds)
            out.append("    long long N, long long ld, const double* t, int t_stride, const double* q, const double* x,")
            out.append("    const double* y, const double* x0, const unsigned* active0, double* sol, int* status,")
            out.append("    unsigned* active, int max_iter) {")
            out.append("  clik::pdl_launch_dependents();")
            out.append("  clik::pdl_wait();   // reads the status[] / active[] the fast pass wrote")
            out.append("  clik::qp_step_tail<Skill>(N, ld, t, t_stride, q, x, y, x0, active0, sol, status, active, max_iter);")
            out.append("}")
            # the same tail pass capped to 4 CTAs per SM (128 registers, the iteration spills): chosen by the
            # host for batches with more tail tiles than the uncapped kernel keeps resident — there the
            # tail is a throughput problem (more CTAs in flight, and its CTAs fit the hole a finished fast-pass
            # CTA of another stream leaves), for small batches it is the latency of the slowest instance
            tcap = int(os.environ.get("CLIK_QP_TAIL_CAP", "4"))
            meta["qp_tail_cap"] = tcap
            if tcap > 0:
                out.append('extern "C" __global__ void __launch_bounds__(%d, %d) clik_qp_tail_capped_kernel(' % (block_threads, tcap))
                out.append("    long long N, long long ld, const double* t, int t_stride, const double* q, const double* x,")
                out.append("    const double* y, const double* x0, const unsigned* active0, double* sol, int* status,")
                out.append("    unsigned* active, int max_iter) {")
                out.append("  clik::pdl_launch_dependents();")
                out.append("  clik::pdl_wait();")
                out.append("  clik::qp_step_tail<Skill>(N, ld, t, t_stride, q, x, y, x0, active0, sol, status, active, max_iter);")
                out.append("}")
    qp_rollout = qp is not None and getattr(qp, "emit_rollout", True)
    if qp_rollout:
        out.append('extern "C" __global__ void __launch_bounds__(%d) clik_qp_rollout_kernel(' % block_threads)
        out.append("    long long N, long long ld, int steps, double dt, const double* t0, int t_stride, double* q, double* x,")
        out.append("    const double* y, double vmax_q, double vmax_x, double* sol_last, int* n_failed, int max_iter) {")
        out.append("  clik::qp_rollout<Skill>(N, ld, steps, dt, t0, t_stride, q, x, y, vmax_q, vmax_x, sol_last, n_failed,")
        out.append("                          max_iter);")
        out.append("}")
    out.append('extern "C" __global__ void clik_sizes_kernel(int* o) {')
    flags = 0
    if pinv is not None:
        flags |= 2 | (1 if meta.get("pinv_staged_kernel") else 0)
        flags |= (32 if meta.get("pinv_group") else 0) | (64 if meta.get("pinv_split") else 0)
    if qp is not None:
        flags |= (4 if qp_rollout else 0) | (16 if meta.get("qp_split") else 0)
        flags |= 128 if (meta.get("qp_split") and meta.get("qp_tail_cap", 0) > 0) else 0
    out.append("  // manifest: sizes, unroll, optional-kernel flags (1 pinv TMA, 2 pinv rollout, 4 QP rollout, 16 QP fast + tail pair,")
    out.append("  // 32 pinv group kernel, 64 pinv fast kernel, 128 capped QP tail kernel); o[16] statically compiled modes, o[17] block size of the group kernel")
    out.append("  o[0] = %d; o[1] = %d; o[2] = %d; o[3] = %d; o[4] = %d; o[5] = %d; o[6] = %d; o[7] = %d;"
               % (nq, nxv, ny, meta["n_modes"], meta["qp_n"], meta["qp_m"], meta.get("pinv_unroll", 1), flags))
    full = (1, 0xffffffff, 0xffffffff, 0xffffffff)
    pm, qm = meta.get("pinv_read_masks", full), meta.get("qp_read_masks", full)
    out.append("  // input rows the kernels read (t, q, x, y bit masks): pinv then QP")
    out.append("  " + " ".join("o[%d] = (int)0x%xu;" % (8 + k, v) for k, v in enumerate(tuple(pm) + tuple(qm))))
    out.append("  o[16] = %d; o[17] = %s;" % (meta.get("pinv_static_modes", 1),
                                             "clik::GroupGeometry<Skill>::BLOCK" if meta.get("pinv_group") else "0"))
    meta["duals"] = qp is not None and 0 < qp.m <= DUALS_MAX_ROWS
    if meta["duals"]:
        out.append("  o[18] = 1;   // multiplier kernels (1 QP, 2 NLP)")
    meta["vjp"] = bool(vjp) and meta["duals"]
    if meta["vjp"]:
        out.append(_VJP_MANIFEST % 1)
    out.append("}")
    if meta["duals"]:
        out += _emit_qp_duals(qp, sig, sincos_name, block_threads, meta["qp_structured"])
    if meta["vjp"]:
        out += _emit_vjp(qp, "qp", sig, sincos_name, block_threads,
                         "SkillDuals" if meta["qp_structured"] else "Skill", meta["qp_read_masks"], meta)
    return "\n".join(out) + "\n", meta


#: the working-set masks of the step kernels describe rows below 32 only (clik_duals.cuh)
DUALS_MAX_ROWS = 32


def _emit_qp_duals(qp, sig, sincos_name, block_threads, structured):
    """clik_qp_duals_kernel, appended after the manifest so that nothing emitted before changes.  A structured
    skill (eval_qps: dense rows + unit rows, 1/sqrt(h)) also gets the dense eval_qp the kernel reads, in a struct
    derived from Skill; its constants are literals, so the constant bank of the step kernels stays as it is."""
    out = ["", "// ---- constraint multipliers of the step's output (clik_duals.cuh) ----",
           '#include "clik_duals.cuh"']
    skill = "Skill"
    if structured:
        skill = "SkillDuals"
        em = Emitter(qp.syms.names, None, sincos_name)
        for r in range(qp.m):
            for j in range(qp.nx):
                em.assign("d.A[%d]" % (r * qp.nx + j), qp.A[r][j])
            em.assign("d.lb[%d]" % r, qp.lb[r])
            em.assign("d.ub[%d]" % r, qp.ub[r])
        for j in range(qp.nx):
            em.assign("d.h[%d]" % j, qp.h[j])
        out.append("struct SkillDuals : Skill {")
        out.append("  __device__ static __forceinline__ void eval_qp(%s, clik::QpData<SkillDuals>& d) {" % sig)
        out += ["    " + ln for ln in em.finish()]
        out.append("  }")
        out.append("};")
    out.append('extern "C" __global__ void __launch_bounds__(%d) clik_qp_duals_kernel(' % block_threads)
    out.append("    long long N, long long ld, const double* t, int t_stride, const double* q, const double* x,")
    out.append("    const double* y, const double* sol, const int* status, const unsigned* active, double* lam) {")
    out.append("  clik::qp_duals<%s>(N, ld, t, t_stride, q, x, y, sol, status, active, lam);" % skill)
    out.append("}")
    return out


_VJP_MANIFEST = "  o[19] = %d;   // VJP kernels (1 QP, 2 NLP)"


def _emit_vjp(prog, kind, sig, sincos_name, block_threads, base, base_masks, meta):
    """clik_<kind>_vjp_kernel (clik_vjp.cuh), appended after the multiplier kernel: a struct derived from `base`
    (the struct whose eval_qp / eval_nlp_pre the multiplier kernel reads) adds eval_vjp, the gradient program of
    Phi (codegen/vjp.py), and the rows the kernel loads (those of `base_masks` and those eval_vjp reads).  Its
    constants are literals, so the constant bank of the step kernels stays as it is."""
    from .vjp import VjpProgram
    vp = VjpProgram(prog, kind)
    em = Emitter(vp.names, None, sincos_name)
    em.assign("tb", vp.t)
    for arr, nodes in (("qb", vp.q), ("xb", vp.x), ("yb", vp.y)):
        for j, n in enumerate(nodes):
            em.assign("%s[%d]" % (arr, j), n)
    masks = tuple(a | b for a, b in zip(base_masks, em.read_masks(prog.syms)))
    meta["vjp_eval"] = em.counts()
    meta["vjp_read_masks"] = masks
    n, m = prog.nx, prog.m
    out = ["", "// ---- reverse-mode derivative of the step's output (clik_vjp.cuh) ----",
           '#include "clik_vjp.cuh"',
           "struct SkillVjp : %s {" % base,
           "  using Base = %s;   // the struct whose row evaluation the kernel calls" % base,
           "  static constexpr unsigned VJP_READ_T = %du, VJP_READ_Q = 0x%xu, VJP_READ_X = 0x%xu, VJP_READ_Y = 0x%xu;"
           % masks,
           "  __device__ static __forceinline__ void eval_vjp(%s," % sig,
           "      const double (&xs_)[%d], const double (&lam_)[%d], const double (&u_)[%d], const double (&vu_)[%d],"
           % (n, m, n, m),
           "      const double (&vl_)[%d], double& tb, double (&qb)[%d], double (&xb)[%d], double (&yb)[%d]) {"
           % (m, max(prog.n_rob, 1), max(prog.n_virt, 1), max(prog.n_in, 1))]
    out += ["    " + ln for ln in em.finish()]
    out += ["  }",
            "};",
            'extern "C" __global__ void __launch_bounds__(%d) clik_%s_vjp_kernel(' % (block_threads, kind),
            "    long long N, long long ld, const double* t, int t_stride, const double* q, const double* x,",
            "    const double* y, const double* sol, const int* status, const unsigned* active, const double* sol_bar,",
            "    double* t_bar, double* q_bar, double* x_bar, double* y_bar) {",
            "  clik::%s_vjp<SkillVjp>(N, ld, t, t_stride, q, x, y, sol, status, active, sol_bar, t_bar, q_bar, x_bar,"
            % kind,
            "                         y_bar);",
            "}"]
    return out


def nlp_hoisted(nlp):
    """The maximal decision-free subexpressions the cost graph (F, g, H) consumes: every non-constant
    argument without a decision symbol below it of a node that has one, and every output without one.
    eval_nlp_pre computes them once per step; the SQP iteration only reads them."""
    dec = {n.id for n in nlp.dec}
    outs = [nlp.F] + list(nlp.g) + list(nlp.H)
    dep = {}
    for n in dag.topo(outs):
        dep[n.id] = n.id in dec or any(dep[a.id] for a in n.args)
    P, seen = [], set()

    def want(n):
        if n.op != "const" and not dep[n.id] and n.id not in seen:
            seen.add(n.id)
            P.append(n)
    for n in dag.topo(outs):
        if dep[n.id]:
            for a in n.args:
                want(a)
    for o in outs:
        want(o)
    return P


def _emit_nlp(nlp, label, block_threads, tol, vjp=False):
    """Translation unit of the reactive-NLP controller (csrc/clik_nlp.cuh instantiated on the skill)."""
    const_table = [] if os.environ.get("CLIK_CONSTBANK", "1") == "1" else None
    sincos_name = "clik::sincos_fast" if os.environ.get("CLIK_FAST_SINCOS", "1") == "1" else "sincos"
    nq, nxv, ny, nx, m = nlp.n_rob, nlp.n_virt, nlp.n_in, nlp.nx, nlp.m
    P = nlp_hoisted(nlp)
    npar = len(P)
    meta = {"label": label, "n_robot": nq, "n_virtual": nxv, "n_input": ny,
            "has_pinv": False, "has_qp": False, "has_nlp": True,
            "n_modes": 1, "qp_n": nx, "qp_m": m, "block_threads": block_threads,
            "nlp_quadratic": bool(nlp.quadratic), "nlp_hoisted": npar, "nlp_tol": float(tol)}
    out = ["// generated by casclik_b200.codegen for skill %r -- do not edit" % label,
           '#include "clik_math.cuh"',
           '#include "clik_qp.cuh"',
           '#include "clik_nlp.cuh"',
           ""]
    pre_struct = []
    struct_at = len(out)
    out.append("struct Skill {")
    out.append("  static constexpr int NQ = %d, NX = %d, NY = %d, NS = %d;" % (nq, nxv, ny, nq + nxv))
    out.append("  static constexpr int BLOCK = %d;   // threads per CTA of the step kernels" % block_threads)
    out.append("  static constexpr int NN = %d, NM = %d, NP = %d;   // decision variables, rows, hoisted values"
               % (nx, m, npar))
    out.append("  static constexpr bool NLP_QUADRATIC = %s;   // Hessian free of decision variables: one subproblem"
               % ("true" if nlp.quadratic else "false"))
    out.append("  static constexpr double NLP_TOL = %s;" % literal(float(tol)))
    out.append("  static constexpr int NLP_QP_ITER = %d;   // iteration cap of each subproblem" % (10 * (nx + m)))
    sig = ("const double t, const double (&q)[%d], const double (&x)[%d], const double (&y)[%d]"
           % (max(nq, 1), max(nxv, 1), max(ny, 1)))
    # once per step: the constraint rows and the hoisted values
    em = Emitter(nlp.syms.names, const_table, sincos_name)
    for r in range(m):
        for j in range(nx):
            em.assign("d.A[%d]" % (r * nx + j), nlp.A[r][j])
        em.assign("d.lb[%d]" % r, nlp.lb[r])
        em.assign("d.ub[%d]" % r, nlp.ub[r])
    for k, n in enumerate(P):
        em.assign("d.P[%d]" % k, n)
    out.append("  __device__ static __forceinline__ void eval_nlp_pre(%s, clik::NlpData<Skill>& d) {" % sig)
    out += ["    " + ln for ln in em.finish()]
    out.append("  }")
    meta["nlp_read_masks"] = em.read_masks(nlp.syms)
    pre_counts = em.counts()
    # per SQP iteration / line-search trial: F (and g, H) from the decision variables and the hoisted values
    dec_names = {n.id: "v[%d]" % j for j, n in enumerate(nlp.dec)}
    leaves = {n.id: "P[%d]" % k for k, n in enumerate(P)}
    psig = "const double (&P)[%d], const double (&v)[%d]" % (max(npar, 1), nx)
    emf = Emitter(dec_names, const_table, sincos_name, leaves=leaves)
    emf.assign("f_", nlp.F)
    out.append("  __device__ static __forceinline__ double eval_nlp_f(%s) {" % psig)
    out.append("    double f_;")
    out += ["    " + ln for ln in emf.finish()]
    out.append("    return f_;")
    out.append("  }")
    emg = Emitter(dec_names, const_table, sincos_name, leaves=leaves)
    emg.assign("f_", nlp.F)
    for j in range(nx):
        emg.assign("g[%d]" % j, nlp.g[j])
    for k, n in enumerate(nlp.H):
        emg.assign("H[%d]" % k, n)
    out.append("  __device__ static __forceinline__ double eval_nlp_fgH(%s, double (&g)[%d], double (&H)[%d]) {"
               % (psig, nx, nx * (nx + 1) // 2))
    out.append("    double f_;")
    out += ["    " + ln for ln in emg.finish()]
    out.append("    return f_;")
    out.append("  }")
    meta["nlp_eval"] = {"pre": pre_counts, "f": emf.counts(), "fgH": emg.counts()}
    out.append("  static constexpr unsigned NLP_READ_T = %du, NLP_READ_Q = 0x%xu, NLP_READ_X = 0x%xu, NLP_READ_Y = 0x%xu;"
               % meta["nlp_read_masks"])
    meta["nlp_inputs_read"] = em.inputs_read()
    out.append("};")
    out.append("")
    if const_table:
        pre_struct.append("__constant__ double KC[%d] = {%s};" % (
            len(const_table), ", ".join(literal(v) for v in const_table)))
    out[struct_at:struct_at] = pre_struct
    out.append('extern "C" __global__ void __launch_bounds__(%d) clik_nlp_kernel(' % block_threads)
    out.append("    long long N, long long ld, const double* t, int t_stride, const double* q, const double* x,")
    out.append("    const double* y, const double* x0, double* sol, int* status, int* iters, unsigned* active,")
    out.append("    int max_iter) {")
    out.append("  clik::nlp_step<Skill>(N, ld, t, t_stride, q, x, y, x0, sol, status, iters, active, max_iter);")
    out.append("}")
    out.append('extern "C" __global__ void __launch_bounds__(%d) clik_nlp_rollout_kernel(' % block_threads)
    out.append("    long long N, long long ld, int steps, double dt, const double* t0, int t_stride, double* q, double* x,")
    out.append("    const double* y, double vmax_q, double vmax_x, double* sol_last, int* n_failed, int max_iter) {")
    out.append("  clik::nlp_rollout<Skill>(N, ld, steps, dt, t0, t_stride, q, x, y, vmax_q, vmax_x, sol_last, n_failed,")
    out.append("                           max_iter);")
    out.append("}")
    out.append('extern "C" __global__ void clik_sizes_kernel(int* o) {')
    out.append("  // manifest: sizes (o[4], o[5]: NLP variables and rows), flags (256 NLP step + rollout kernels)")
    out.append("  o[0] = %d; o[1] = %d; o[2] = %d; o[3] = 1; o[4] = %d; o[5] = %d; o[6] = 1; o[7] = 256;"
               % (nq, nxv, ny, nx, m))
    full = (1, 0xffffffff, 0xffffffff, 0xffffffff)
    out.append("  // input rows the kernels read (t, q, x, y bit masks): (no pinv kernel) then NLP")
    out.append("  " + " ".join("o[%d] = (int)0x%xu;" % (8 + k, v) for k, v in enumerate(full + tuple(meta["nlp_read_masks"]))))
    out.append("  o[16] = 1; o[17] = 0;")
    meta["duals"] = 0 < m <= DUALS_MAX_ROWS
    if meta["duals"]:
        out.append("  o[18] = 2;   // multiplier kernels (1 QP, 2 NLP)")
    meta["vjp"] = bool(vjp) and meta["duals"]
    if meta["vjp"]:
        out.append(_VJP_MANIFEST % 2)
    out.append("}")
    if meta["duals"]:
        out += ["", "// ---- constraint multipliers of the step's output (clik_duals.cuh) ----",
                '#include "clik_duals.cuh"',
                'extern "C" __global__ void __launch_bounds__(%d) clik_nlp_duals_kernel(' % block_threads,
                "    long long N, long long ld, const double* t, int t_stride, const double* q, const double* x,",
                "    const double* y, const double* sol, const int* status, const unsigned* active, double* lam) {",
                "  clik::nlp_duals<Skill>(N, ld, t, t_stride, q, x, y, sol, status, active, lam);",
                "}"]
    if meta["vjp"]:
        out += _emit_vjp(nlp, "nlp", sig, sincos_name, block_threads, "Skill", meta["nlp_read_masks"], meta)
    return "\n".join(out) + "\n", meta


def emit_c_function(name, sym_names, outputs, arg_decl):
    """Plain C version of a node list (tests: gcc-compiled text vs NumPy interpreter)."""
    em = Emitter(sym_names)
    for i, n in enumerate(outputs):
        em.assign("out[%d]" % i, n)
    lines = ["#include <math.h>",
             "static void sincos_(double a, double* s, double* c) { *s = sin(a); *c = cos(a); }",
             "#define sincos sincos_",
             "void %s(%s, double* out) {" % (name, arg_decl)]
    lines += ["  " + ln for ln in em.finish()]
    lines.append("}")
    return "\n".join(lines) + "\n"
