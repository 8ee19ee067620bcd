"""Minimal dimod-compatible ``ConstrainedQuadraticModel`` for the calls at CQM_clustering.py:30-48, 62-84:
``dimod.Binary(label)`` arithmetic, ``cqm.add_discrete(labels, label=)``, ``cqm.set_objective(expr)``,
``cqm.add_constraint(expr >= c, label=)``.

``to_lowered`` turns the constraints into penalties (the reference leaves that to LeapHybridCQMSampler):
one-hot groups -> A*(sum x - 1)^2; linear (in)equalities -> dimod's binary-slack penalty with multiplier B.
For graphs of benchmark size use ``models.cqm_model`` (vectorised, rank-1 structured) instead.
"""
from __future__ import annotations

from typing import Dict, Hashable, List, Optional, Tuple

import numpy as np

from .bqm import BinaryQuadraticModel
from .models import Groups, LoweredModel, lowered_from_bqm


class QuadExpr:
    """offset + sum linear[v] v + sum quadratic[(u, v)] u v over binary variables."""

    __slots__ = ("linear", "quadratic", "offset")

    def __init__(self, linear=None, quadratic=None, offset=0.0):
        self.linear: Dict[Hashable, float] = dict(linear or {})
        self.quadratic: Dict[Tuple[Hashable, Hashable], float] = dict(quadratic or {})
        self.offset = float(offset)

    def copy(self):
        return QuadExpr(self.linear, self.quadratic, self.offset)

    def _iadd(self, other, sign=1.0):
        if isinstance(other, QuadExpr):
            for v, b in other.linear.items():
                self.linear[v] = self.linear.get(v, 0.0) + sign * b
            for k, b in other.quadratic.items():
                if k not in self.quadratic and (k[1], k[0]) in self.quadratic:
                    k = (k[1], k[0])
                self.quadratic[k] = self.quadratic.get(k, 0.0) + sign * b
            self.offset += sign * other.offset
        else:
            self.offset += sign * float(other)
        return self

    def __add__(self, other):
        return self.copy()._iadd(other)

    __radd__ = __add__

    def __iadd__(self, other):
        return self._iadd(other)

    def __sub__(self, other):
        return self.copy()._iadd(other, -1.0)

    def __rsub__(self, other):
        return (-self)._iadd(other)

    def __neg__(self):
        return self * -1.0

    def __mul__(self, other):
        if isinstance(other, QuadExpr):
            if self.quadratic or other.quadratic:
                raise ValueError("products of degree > 2 are not representable")
            out = QuadExpr(offset=self.offset * other.offset)
            for v, b in self.linear.items():
                out.linear[v] = out.linear.get(v, 0.0) + b * other.offset
            for v, b in other.linear.items():
                out.linear[v] = out.linear.get(v, 0.0) + b * self.offset
            for u, a in self.linear.items():
                for v, b in other.linear.items():
                    if u == v:  # x*x = x for binaries
                        out.linear[u] = out.linear.get(u, 0.0) + a * b
                    else:
                        k = (u, v) if (v, u) not in out.quadratic else (v, u)
                        out.quadratic[k] = out.quadratic.get(k, 0.0) + a * b
            return out
        c = float(other)
        return QuadExpr({v: b * c for v, b in self.linear.items()}, {k: b * c for k, b in self.quadratic.items()},
                        self.offset * c)

    __rmul__ = __mul__

    def __ge__(self, rhs):
        return Constraint(self - rhs, ">=")

    def __le__(self, rhs):
        return Constraint(self - rhs, "<=")

    def __eq__(self, rhs):  # noqa: A003 - comparison builds a constraint, as in dimod
        return Constraint(self - rhs, "==")

    __hash__ = None

    def energies(self, samples: np.ndarray, index: Dict[Hashable, int]) -> np.ndarray:
        S = np.atleast_2d(samples).astype(np.float64)
        e = np.full(S.shape[0], self.offset)
        for v, b in self.linear.items():
            e += b * S[:, index[v]]
        for (u, v), b in self.quadratic.items():
            e += b * S[:, index[u]] * S[:, index[v]]
        return e


class Constraint:
    """``lhs (sense) 0`` with lhs a QuadExpr whose offset carries -rhs."""

    def __init__(self, lhs: QuadExpr, sense: str):
        self.lhs = lhs
        self.sense = sense


def Binary(label: Hashable) -> QuadExpr:
    return QuadExpr({label: 1.0})


class ConstrainedQuadraticModel:
    def __init__(self):
        self.objective = QuadExpr()
        self.constraints: Dict[Hashable, Constraint] = {}
        self.discrete: Dict[Hashable, List[Hashable]] = {}
        self.variables: List[Hashable] = []
        self._seen = set()

    def _touch(self, labels):
        for v in labels:
            if v not in self._seen:
                self._seen.add(v)
                self.variables.append(v)

    def set_objective(self, expr):
        if not isinstance(expr, QuadExpr):
            expr = QuadExpr(offset=float(expr))
        self.objective = expr
        self._touch(expr.linear.keys())
        for u, v in expr.quadratic.keys():
            self._touch((u, v))

    def add_discrete(self, labels, label: Optional[Hashable] = None):
        labels = list(labels)
        if label is None:
            label = f"discrete_{len(self.discrete)}"
        if label in self.discrete or label in self.constraints:
            raise ValueError(f"a constraint labelled {label!r} already exists")
        for grp in self.discrete.values():
            if set(grp) & set(labels):
                raise ValueError("discrete constraints must be disjoint")
        self.discrete[label] = labels
        self._touch(labels)
        return label

    def add_constraint(self, constraint: Constraint, label: Optional[Hashable] = None):
        if not isinstance(constraint, Constraint):
            raise TypeError("expected a comparison such as `expr >= 20`")
        if constraint.lhs.quadratic:
            raise ValueError("only linear constraints can be lowered to slack penalties")
        if label is None:
            label = f"c{len(self.constraints)}"
        if label in self.discrete or label in self.constraints:
            raise ValueError(f"a constraint labelled {label!r} already exists")
        self.constraints[label] = constraint
        self._touch(constraint.lhs.linear.keys())
        return label

    def check_feasible(self, samples: np.ndarray, labels: List[Hashable]) -> np.ndarray:
        index = {v: i for i, v in enumerate(labels)}
        S = np.atleast_2d(samples)
        ok = np.ones(S.shape[0], dtype=bool)
        for grp in self.discrete.values():
            ok &= S[:, [index[v] for v in grp]].sum(axis=1) == 1
        for con in self.constraints.values():
            val = con.lhs.energies(S, index)
            if con.sense == ">=":
                ok &= val >= -1e-9
            elif con.sense == "<=":
                ok &= val <= 1e-9
            else:
                ok &= np.abs(val) <= 1e-9
        return ok

    def to_bqm(self, onehot_penalty: float, constraint_penalty: float, constraints: bool = True) -> BinaryQuadraticModel:
        """Objective + one-hot penalties + (``constraints``) slack penalties of the linear constraints."""
        bqm = BinaryQuadraticModel({}, {}, self.objective.offset, "BINARY")
        for v in self.variables:
            bqm.add_variable(v, 0.0)
        for v, b in self.objective.linear.items():
            bqm.add_linear(v, b)
        for (u, v), b in self.objective.quadratic.items():
            bqm.add_quadratic(u, v, b)
        for grp in self.discrete.values():
            bqm.add_linear_equality_constraint([(v, 1) for v in grp], onehot_penalty, -1)
        import warnings
        for label, con in (self.constraints.items() if constraints else ()):
            terms = [(v, int(a) if float(a).is_integer() else a) for v, a in con.lhs.linear.items()]
            const = con.lhs.offset
            const = int(const) if float(const).is_integer() else const
            hi = sum(a for _, a in terms if a > 0) + const
            lo = sum(a for _, a in terms if a < 0) + const
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                if con.sense == "==":
                    bqm.add_linear_equality_constraint(terms, constraint_penalty, const)
                elif con.sense == ">=":
                    bqm.add_linear_inequality_constraint(terms, constraint_penalty, label, constant=const, lb=0, ub=hi)
                else:
                    bqm.add_linear_inequality_constraint(terms, constraint_penalty, label, constant=const, lb=lo, ub=0)
        return bqm

    def default_penalties(self) -> Tuple[float, float]:
        gain: Dict[Hashable, float] = {}
        for v, b in self.objective.linear.items():
            gain[v] = gain.get(v, 0.0) + abs(b)
        for (u, v), b in self.objective.quadratic.items():
            gain[u] = gain.get(u, 0.0) + abs(b)
            gain[v] = gain.get(v, 0.0) + abs(b)
        return max(gain.values(), default=0.0) + 1.0, 1.0

    def to_lowered(self, onehot_penalty: Optional[float] = None, constraint_penalty: Optional[float] = None,
                   lowering: str = "slack") -> LoweredModel:
        """Spin model of the CQM.  ``lowering="slack"``: every linear constraint becomes a slack penalty (dimod's
        add_linear_inequality_constraint).  ``"interval"``: no slack variables; each constraint ``sum a_i x_i + c (sense) 0``
        becomes one interval group (``models.Groups``) with coef a_i, kappa = sum a_i + 2c, lam = B and bounds [0, +inf) for
        ``>=``, (-inf, 0] for ``<=``, [0, 0] for ``==``: the penalty B * violation^2.  It needs integer a_i and 2c, pairwise
        disjoint constraint variables and at most QA_MAX_GROUPS constraints, and raises ValueError otherwise.  Discrete
        (one-hot) constraints are couplers either way."""
        if lowering not in ("slack", "interval"):
            raise ValueError(f"lowering must be 'slack' or 'interval', not {lowering!r}")
        A0, B0 = self.default_penalties()
        A = A0 if onehot_penalty is None else float(onehot_penalty)
        B = B0 if constraint_penalty is None else float(constraint_penalty)
        interval = lowering == "interval"
        if interval:
            groups_spec = self._interval_groups()
        model = lowered_from_bqm(self.to_bqm(A, B, constraints=not interval))
        if interval:
            index = {v: i for i, v in enumerate(model.labels)}
            n, G = model.num_variables, len(groups_spec)
            grp = np.full(n, -1, dtype=np.int32)
            coef = np.zeros(n, dtype=np.int32)
            kappa, lo, hi = (np.zeros(G, dtype=np.int64) for _ in range(3))
            for g, (terms, kap, lo_g, hi_g) in enumerate(groups_spec):
                for v, a in terms:
                    grp[index[v]], coef[index[v]] = g, a
                kappa[g], lo[g], hi[g] = kap, lo_g, hi_g
            model.groups = Groups(grp, coef, np.full(G, B), kappa, lo, hi)
        model.meta.update({"kind": "cqm_generic", "cqm": self, "onehot_penalty": A, "size_penalty": B, "lowering": lowering})
        return model

    def _interval_groups(self):
        """[(terms [(label, int a)], kappa, lo, hi)] of the non-discrete constraints, or ValueError."""
        from ._lib import QA_MAX_GROUPS
        if len(self.constraints) > QA_MAX_GROUPS:
            raise ValueError(f"{len(self.constraints)} constraints: the interval lowering takes at most {QA_MAX_GROUPS}")
        owner: Dict[Hashable, Hashable] = {}
        out = []
        i64 = np.iinfo(np.int64)
        for label, con in self.constraints.items():
            terms = []
            for v, a in con.lhs.linear.items():
                if not float(a).is_integer():
                    raise ValueError(f"constraint {label!r}: coefficient {a} of {v!r} is not an integer")
                if v in owner:
                    raise ValueError(f"variable {v!r} appears in constraints {owner[v]!r} and {label!r}: interval groups "
                                     "must not overlap")
                owner[v] = label
                terms.append((v, int(a)))
            c2 = 2 * con.lhs.offset
            if not float(c2).is_integer():
                raise ValueError(f"constraint {label!r}: twice its constant ({c2}) is not an integer")
            kap = sum(a for _, a in terms) + int(c2)
            lo, hi = {">=": (0, i64.max), "<=": (i64.min, 0), "==": (0, 0)}[con.sense]
            out.append((terms, kap, lo, hi))
        return out
