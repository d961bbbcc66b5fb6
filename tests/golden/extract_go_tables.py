#!/usr/bin/env python3
"""Extract the reference's table-driven test vectors into JSON golden fixtures.

Run it against a checkout of armadaproject/armada; the JSON it writes is committed under
tests/golden/ and is all the tests read:

    python tests/golden/extract_go_tables.py <path to the armada checkout>

The Go test files declare their known-answer tables as composite literals
(`tests := map[string]struct{...}{ "name": {Field: expr, ...}, ... }`).  This script parses
that literal with a small recursive-descent parser for the subset of Go expression syntax
the tables use and stores a neutral AST:

    {"lit": "<go type>", "elems": [[key|null, value], ...]}   composite literal
    {"call": "pkg.Fn", "args": [...]}                          function call
    {"id": "pkg.Name"}                                         identifier
    {"op": "/", "l": ..., "r": ...} / {"neg": ...}             arithmetic
    plain JSON numbers / strings / bools / null                literals
    {"unsupported": "<why>"}                                   closures etc. (case is skipped)

tests/go_tables.py evaluates the AST against the Python fixtures (tests/fixtures.py).
Nothing but DATA (inputs + expected answers) is extracted; no reference code is copied.
"""
from __future__ import annotations

import json
import os
import re
import sys

REF = os.path.join(sys.argv[1] if len(sys.argv) > 1 else ".", "internal", "scheduler")
OUT = os.path.dirname(os.path.abspath(__file__))

TABLES = [
    # (output name, go file, start marker regex (the table variable declaration))
    ("preempting_queue_scheduler", "scheduling/preempting_queue_scheduler_test.go", r"func TestPreemptingQueueScheduler\(", r"tests := map\[string\]struct \{"),
    ("queue_scheduler", "scheduling/queue_scheduler_test.go", r"func TestQueueScheduler\(", r"tests := map\[string\]struct \{"),
    ("gang_scheduler", "scheduling/gang_scheduler_test.go", r"func TestGangScheduler\(", r"tests := map\[string\]struct \{"),
    ("node_type_iterator", "nodedb/nodeiteration_test.go", r"func TestNodeTypeIterator\(", r"tests := map\[string\]struct \{"),
    ("node_types_iterator", "nodedb/nodeiteration_test.go", r"func TestNodeTypesIterator\(", r"tests := map\[string\]struct \{"),
    ("calculate_fair_shares", "scheduling/context/scheduling_test.go", r"func TestCalculateFairShares\(", r"tests := map\[string\]struct \{"),
    ("dominant_resource_fairness", "scheduling/fairness/fairness_test.go", r"func TestDominantResourceFairness\(", r"tests := map\[string\]struct \{"),
    ("schedule_individually", "nodedb/nodedb_test.go", r"func TestScheduleIndividually\(", r"tests := map\[string\]struct \{"),
    ("schedule_many", "nodedb/nodedb_test.go", r"func TestScheduleMany\(", r"tests := map\[string\]struct \{"),
]

TOKEN_RE = re.compile(
    r"""
    (?P<ws>\s+)
  | (?P<lcomment>//[^\n]*)
  | (?P<bcomment>/\*.*?\*/)
  | (?P<float>\d[\d_]*\.\d*(?:[eE][+-]?\d+)?|\.\d+(?:[eE][+-]?\d+)?|\d+[eE][+-]?\d+)
  | (?P<int>0[xX][0-9a-fA-F_]+|\d[\d_]*)
  | (?P<str>"(?:\\.|[^"\\])*")
  | (?P<raw>`[^`]*`)
  | (?P<ident>[A-Za-z_][A-Za-z0-9_]*)
  | (?P<op>:=|\.\.\.|<<|>>|&&|\|\||==|!=|<=|>=|[{}()\[\],:.*&+\-/;=<>!|%])
""",
    re.X | re.S,
)


class Unsupported(Exception):
    pass


def tokenize(src: str):
    toks = []
    pos = 0
    while pos < len(src):
        m = TOKEN_RE.match(src, pos)
        if not m:
            raise SyntaxError(f"cannot tokenize at {pos}: {src[pos:pos+40]!r}")
        pos = m.end()
        kind = m.lastgroup
        if kind in ("ws", "lcomment", "bcomment"):
            continue
        toks.append((kind, m.group()))
    return toks


class Parser:
    def __init__(self, toks):
        self.t = toks
        self.i = 0

    def peek(self, k=0):
        return self.t[self.i + k] if self.i + k < len(self.t) else ("eof", "")

    def next(self):
        tok = self.peek()
        self.i += 1
        return tok

    def accept(self, val):
        if self.peek()[1] == val:
            self.i += 1
            return True
        return False

    def expect(self, val):
        tok = self.next()
        if tok[1] != val:
            raise SyntaxError(f"expected {val!r} got {tok!r} at token {self.i}")

    # ---- types ----------------------------------------------------------------------------
    def parse_type(self) -> str:
        k, v = self.peek()
        if v == "[":
            self.next()
            inner = ""
            while self.peek()[1] != "]":
                inner += self.next()[1]
            self.expect("]")
            return "[" + inner + "]" + self.parse_type()
        if v == "map":
            self.next()
            self.expect("[")
            key = self.parse_type()
            self.expect("]")
            return "map[" + key + "]" + self.parse_type()
        if v == "*":
            self.next()
            return "*" + self.parse_type()
        if v == "struct":
            self.next()
            self.skip_braces()
            return "struct{}"
        if v == "func":
            raise Unsupported("func type")
        if k == "ident":
            name = self.next()[1]
            while self.peek()[1] == "." and self.peek(1)[0] == "ident":
                self.next()
                name += "." + self.next()[1]
            if self.peek()[1] == "[":  # generic instantiation, e.g. foo[T]
                raise Unsupported("generic type")
            return name
        raise SyntaxError(f"bad type at {self.peek()!r}")

    def skip_braces(self):
        self.expect("{")
        depth = 1
        while depth:
            v = self.next()[1]
            if v == "{":
                depth += 1
            elif v == "}":
                depth -= 1

    # ---- expressions ----------------------------------------------------------------------
    def parse_expr(self):
        left = self.parse_term()
        while self.peek()[1] in ("+", "-"):
            op = self.next()[1]
            right = self.parse_term()
            left = {"op": op, "l": left, "r": right}
        return left

    def parse_term(self):
        left = self.parse_unary()
        while self.peek()[1] in ("*", "/"):
            op = self.next()[1]
            right = self.parse_unary()
            left = {"op": op, "l": left, "r": right}
        return left

    def parse_unary(self):
        v = self.peek()[1]
        if v == "-":
            self.next()
            return {"neg": self.parse_unary()}
        if v == "&":
            self.next()
            return self.parse_unary()
        return self.parse_primary()

    def parse_composite_body(self, typ: str):
        self.expect("{")
        elems = []
        while self.peek()[1] != "}":
            key = None
            if self.peek()[1] == "{":
                val = self.parse_composite_body("")
            else:
                val = self.parse_expr()
            if self.accept(":"):
                key = val
                if self.peek()[1] == "{":
                    val = self.parse_composite_body("")
                else:
                    val = self.parse_expr()
            elems.append([key, val])
            if not self.accept(","):
                break
        self.expect("}")
        return {"lit": typ, "elems": elems}

    def parse_primary(self):
        k, v = self.peek()
        if v == "func":
            # closure: skip "func(...) T { ... }" and an optional call "()"
            self.skip_func()
            return {"unsupported": "closure"}
        if v in ("[", "map", "struct") or (v == "*" and self.peek(1)[1] in ("[", "map")):
            typ = self.parse_type()
            if self.peek()[1] == "{":
                return self.parse_composite_body(typ)
            if self.peek()[1] == "(":  # conversion, e.g. []byte("x")
                self.next()
                inner = self.parse_expr()
                self.expect(")")
                return {"call": typ, "args": [inner]}
            raise SyntaxError(f"type {typ} not followed by literal")
        if v == "(":
            self.next()
            e = self.parse_expr()
            self.expect(")")
            return self.parse_suffix(e)
        if k == "int":
            self.next()
            return int(v.replace("_", ""), 0)
        if k == "float":
            self.next()
            return float(v.replace("_", ""))
        if k == "str":
            self.next()
            return json.loads(v)
        if k == "raw":
            self.next()
            return v[1:-1]
        if k == "ident":
            name = self.next()[1]
            if name in ("true", "false"):
                return name == "true"
            if name == "nil":
                return None
            while self.peek()[1] == "." and self.peek(1)[0] == "ident":
                self.next()
                name += "." + self.next()[1]
            node = {"id": name}
            if self.peek()[1] == "{":
                return self.parse_composite_body(name)
            return self.parse_suffix(node)
        raise SyntaxError(f"unexpected token {self.peek()!r} at {self.i}")

    def parse_suffix(self, node):
        while True:
            v = self.peek()[1]
            if v == "(":
                self.next()
                args = []
                while self.peek()[1] != ")":
                    args.append(self.parse_expr())
                    if self.accept("..."):
                        pass
                    if not self.accept(","):
                        break
                self.expect(")")
                name = node["id"] if isinstance(node, dict) and "id" in node else None
                node = {"call": name, "args": args} if name else {"callexpr": node, "args": args}
            elif v == "[":
                self.next()
                if self.peek()[1] == ":":
                    self.next()
                    hi = self.parse_expr()
                    self.expect("]")
                    node = {"slice": node, "lo": None, "hi": hi}
                else:
                    idx = self.parse_expr()
                    if self.accept(":"):
                        hi = None if self.peek()[1] == "]" else self.parse_expr()
                        self.expect("]")
                        node = {"slice": node, "lo": idx, "hi": hi}
                    else:
                        self.expect("]")
                        node = {"index": node, "i": idx}
            elif v == "." and self.peek(1)[0] == "ident":
                self.next()
                node = {"sel": node, "name": self.next()[1]}
            else:
                return node

    def skip_func(self):
        self.expect("func")
        # parameters
        self.expect("(")
        depth = 1
        while depth:
            v = self.next()[1]
            depth += v == "("
            depth -= v == ")"
        while self.peek()[1] != "{":  # result type
            self.next()
        self.skip_braces()
        if self.peek()[1] == "(":
            self.next()
            depth = 1
            while depth:
                v = self.next()[1]
                depth += v == "("
                depth -= v == ")"


def extract(go_path: str, func_re: str, table_re: str):
    src = open(go_path).read()
    m = re.search(func_re, src)
    if not m:
        raise RuntimeError(f"{func_re} not found in {go_path}")
    src = src[m.start():]
    m = re.search(table_re, src)
    if not m:
        raise RuntimeError(f"{table_re} not found after {func_re}")
    toks = tokenize(src[m.start():])
    p = Parser(toks)
    # tests := map[string]struct {...}{ ... }
    p.expect("tests")
    p.expect(":=")
    typ = p.parse_type()
    assert typ.startswith("map[string]"), typ
    p.expect("{")
    cases = {}
    while p.peek()[1] != "}":
        name = json.loads(p.next()[1])
        p.expect(":")
        start = p.i
        try:
            cases[name] = p.parse_composite_body("case")
        except Unsupported as e:  # skip to the matching brace
            p.i = start
            p.skip_braces()
            cases[name] = {"unsupported": str(e)}
        if not p.accept(","):
            break
    return cases


def main():
    if not os.path.isdir(REF):
        print(f"{REF} not present; nothing to do (fixtures are committed)", file=sys.stderr)
        return 0
    for name, rel, func_re, table_re in TABLES:
        cases = extract(os.path.join(REF, rel), func_re, table_re)
        out = os.path.join(OUT, f"{name}.json")
        with open(out, "w") as f:
            json.dump({"source": f"internal/scheduler/{rel}", "cases": cases}, f, separators=(",", ":"), sort_keys=False)
        n_unsup = sum(1 for c in cases.values() if json.dumps(c).find('"unsupported"') >= 0)
        print(f"{name}: {len(cases)} cases ({n_unsup} containing closures) -> {out}")
    return 0


if __name__ == "__main__":
    sys.exit(main())
