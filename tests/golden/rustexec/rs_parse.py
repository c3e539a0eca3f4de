"""Lexer + recursive-descent parser for the subset of Rust the reference's src/talib/*.rs is written in.

TEST INFRASTRUCTURE (golden-vector generation only).  The reference cannot be compiled in this image
(no cargo/rustc, and the snapshot does not type-check: SURVEY.md facts 2-3), so the golden vectors
under tests/golden/ are made by EXECUTING the reference's own source text with the small interpreter
in this directory: this file turns the text into a syntax tree, rs_eval.py walks it, polars_model.py
models the handful of polars / std containers the text touches.  Nothing of the reference's text is
stored in the repo; it is read from a checkout of the original at generation time (rustexec.reference_root).

Supported: `use` (skipped), attributes (skipped), `struct` with named fields, `fn` (also nested),
`let` with patterns / type annotations, `if` / `if let` / `else`, `match` with guards, `while` /
`while let`, `for` over ranges and iterators, `loop`, closures, method chains, `?`, `as` casts, paths with
turbofish, tuples, arrays (`[x; n]`), index expressions, `vec![]` / `izip!()` macros, compound
assignment, `return` / `break` / `continue`.  Not supported (absent from the path): struct literals,
traits / impls, generics on user functions, lifetimes, shifts, labels.

Nodes are plain tuples: (kind, ...).  Every node's kind is listed in rs_eval.py's dispatch table.
"""
from __future__ import annotations

import re

TOKEN_RE = re.compile(r"""
  (?P<ws>\s+|//[^\n]*|/\*.*?\*/)
 |(?P<num>\d[\d_]*(?:\.\d[\d_]*)?(?:[eE][+-]?\d+)?(?:f64|f32|usize|isize|i64|i32|u64|u32|u8|i8)?)
 |(?P<str>"(?:[^"\\]|\\.)*")
 |(?P<id>[A-Za-z_][A-Za-z0-9_]*)
 |(?P<op>\.\.=|::|->|=>|==|!=|<=|>=|&&|\|\||\+=|-=|\*=|/=|%=|\.\.|[-+*/%!&|=<>.,;:()\[\]{}?\#@^])
""", re.X | re.S)

INT_SUFFIX = ("usize", "isize", "i64", "i32", "u64", "u32", "u8", "i8")


class RustSyntaxError(Exception):
    pass


def lex(text: str):
    toks, pos = [], 0
    n = len(text)
    while pos < n:
        m = TOKEN_RE.match(text, pos)
        if not m:
            raise RustSyntaxError(f"cannot lex at {text[pos:pos + 40]!r}")
        pos = m.end()
        kind = m.lastgroup
        if kind == "ws":
            continue
        toks.append((kind, m.group(kind), m.start()))
    toks.append(("eof", "", n))
    return toks


BINARY = {  # operator -> precedence (higher binds tighter)
    "*": 11, "/": 11, "%": 11, "+": 10, "-": 10, "&": 8, "^": 7, "|": 6,
    "==": 5, "!=": 5, "<": 5, ">": 5, "<=": 5, ">=": 5, "&&": 4, "||": 3,
}
ASSIGN = ("=", "+=", "-=", "*=", "/=", "%=")
BLOCKLIKE = ("if", "match", "for", "while", "loop", "block", "iflet", "whilelet")


class Parser:
    def __init__(self, text: str, name: str = "<rust>"):
        self.text, self.name = text, name
        self.t = lex(text)
        self.i = 0

    # ---- token helpers -------------------------------------------------------------------------
    def peek(self, k=0):
        return self.t[self.i + k]

    def at(self, val, k=0):
        tok = self.t[self.i + k]
        return tok[1] == val and tok[0] in ("op", "id")

    def accept(self, val):
        if self.at(val):
            self.i += 1
            return True
        return False

    def expect(self, val):
        if not self.accept(val):
            tok = self.peek()
            line = self.text.count("\n", 0, tok[2]) + 1
            raise RustSyntaxError(f"{self.name}:{line}: expected {val!r}, found {tok[1]!r}")

    def ident(self):
        tok = self.peek()
        if tok[0] != "id":
            line = self.text.count("\n", 0, tok[2]) + 1
            raise RustSyntaxError(f"{self.name}:{line}: expected identifier, found {tok[1]!r}")
        self.i += 1
        return tok[1]

    def line(self):
        return self.text.count("\n", 0, self.peek()[2]) + 1

    # ---- items ---------------------------------------------------------------------------------
    def skip_attr(self):
        # '#' ['!'] '[' ... ']'
        self.expect("#")
        self.accept("!")
        self.expect("[")
        depth = 1
        while depth:
            tok = self.peek()
            self.i += 1
            if tok[1] == "[" and tok[0] == "op":
                depth += 1
            elif tok[1] == "]" and tok[0] == "op":
                depth -= 1

    def parse_file(self):
        """-> dict(fns={name: fn_node}, structs={name: [field, ...]}, uses=[path, ...])"""
        fns, structs, uses = {}, {}, []
        while self.peek()[0] != "eof":
            if self.at("#"):
                self.skip_attr()
                continue
            if self.at("use"):
                self.i += 1
                start = self.i
                while not self.at(";"):
                    self.i += 1
                uses.append("".join(tok[1] for tok in self.t[start:self.i]))
                self.expect(";")
                continue
            self.accept("pub")
            if self.at("("):           # pub(crate)
                while not self.accept(")"):
                    self.i += 1
            if self.at("struct"):
                self.i += 1
                name = self.ident()
                self.expect("{")
                fields = []
                while not self.accept("}"):
                    if self.at("#"):
                        self.skip_attr()
                        continue
                    self.accept("pub")
                    fields.append(self.ident())
                    self.expect(":")
                    self.parse_type()
                    self.accept(",")
                structs[name] = fields
                continue
            if self.at("fn"):
                fn = self.parse_fn()
                fns[fn[1]] = fn
                continue
            raise RustSyntaxError(f"{self.name}:{self.line()}: unsupported item at {self.peek()[1]!r}")
        return {"fns": fns, "structs": structs, "uses": uses}

    def parse_fn(self):
        line = self.line()
        self.expect("fn")
        name = self.ident()
        self.expect("(")
        params = []
        while not self.accept(")"):
            pat = self.parse_pattern()
            self.expect(":")
            ty = self.parse_type()
            params.append((pat, ty))
            self.accept(",")
        ret = None
        if self.accept("->"):
            ret = self.parse_type()
        body = self.parse_block()
        return ("fn", name, params, ret, body, line)

    # ---- types (parsed to a compact description; only the names matter to the evaluator) ---------
    def parse_type(self):
        if self.accept("&"):
            self.accept("mut")
            return ("ref", self.parse_type())
        if self.accept("("):
            parts = []
            while not self.accept(")"):
                parts.append(self.parse_type())
                self.accept(",")
            return ("tuple", parts)
        if self.accept("["):
            inner = self.parse_type()
            if self.accept(";"):
                self.parse_expr()
            self.expect("]")
            return ("slice", inner)
        if self.at("impl") or self.at("dyn"):
            self.i += 1
        segs = [self.ident()]
        args = []
        while True:
            if self.at("<"):
                args = self.parse_generic_args()
            if self.at("::") and (self.peek(1)[0] == "id" or self.at("<", 1)):
                self.i += 1
                if self.at("<"):
                    args = self.parse_generic_args()
                else:
                    segs.append(self.ident())
                continue
            break
        return ("path", segs[-1], args)

    def parse_generic_args(self):
        self.expect("<")
        args = []
        while not self.accept(">"):
            args.append(self.parse_type())
            self.accept(",")
        return args

    # ---- patterns ------------------------------------------------------------------------------
    def parse_pattern(self):
        if self.accept("&"):
            self.accept("mut")
            return self.parse_pattern()            # references are transparent in the model
        if self.accept("mut"):
            return ("pbind", self.ident())
        if self.accept("ref"):
            self.accept("mut")
            return ("pbind", self.ident())
        if self.accept("("):
            parts = []
            while not self.accept(")"):
                parts.append(self.parse_pattern())
                self.accept(",")
            return ("ptuple", parts)
        tok = self.peek()
        if tok[0] == "num" or (self.at("-") and self.peek(1)[0] == "num"):
            neg = self.accept("-")
            v = self.number(self.peek()[1])
            self.i += 1
            return ("plit", -v if neg else v)
        if tok[0] == "id":
            name = self.ident()
            if name == "_":
                return ("pwild",)
            if name == "true" or name == "false":
                return ("plit", name == "true")
            if name == "None":
                return ("pnone",)
            if name in ("Some", "Ok", "Err") and self.accept("("):
                inner = self.parse_pattern()
                self.accept(",")
                self.expect(")")
                return ("pctor", name, inner)
            return ("pbind", name)
        raise RustSyntaxError(f"{self.name}:{self.line()}: unsupported pattern at {tok[1]!r}")

    # ---- blocks and statements -----------------------------------------------------------------
    def parse_block(self):
        """-> ('block', [stmt...], tail_expr | None)"""
        self.expect("{")
        stmts, tail = [], None
        while not self.accept("}"):
            if self.accept(";"):
                continue
            if self.at("#"):
                self.skip_attr()
                continue
            if self.at("let"):
                line = self.line()
                self.i += 1
                pat = self.parse_pattern()
                if self.accept(":"):
                    self.parse_type()
                init = None
                if self.accept("="):
                    init = self.parse_expr()
                self.expect(";")
                stmts.append(("let", pat, init, line))
                continue
            if self.at("fn"):
                stmts.append(("fnitem", self.parse_fn()))
                continue
            if self.at("use"):
                while not self.accept(";"):
                    self.i += 1
                continue
            line = self.line()
            e = self.parse_expr(stmt=True)
            if self.accept(";"):
                stmts.append(("expr", e, line))
            elif self.at("}"):
                tail = e
            elif e[0] in BLOCKLIKE:
                stmts.append(("expr", e, line))
            else:
                raise RustSyntaxError(f"{self.name}:{self.line()}: expected ';' or '}}' after expression, found {self.peek()[1]!r}")
        return ("block", stmts, tail)

    # ---- expressions ---------------------------------------------------------------------------
    def parse_expr(self, stmt=False):
        line = self.line()
        lhs = self.parse_range(stmt)
        if self.peek()[0] == "op" and self.peek()[1] in ASSIGN:
            op = self.peek()[1]
            self.i += 1
            rhs = self.parse_expr()
            return ("assign", op, lhs, rhs, line)
        return lhs

    def parse_range(self, stmt=False):
        if self.at("..") or self.at("..="):
            raise RustSyntaxError(f"{self.name}:{self.line()}: open-start ranges unsupported")
        lhs = self.parse_binary(0, stmt)
        if self.at("..") or self.at("..="):
            incl = self.peek()[1] == "..="
            self.i += 1
            rhs = self.parse_binary(0)
            return ("range", lhs, rhs, incl)
        return lhs

    def parse_binary(self, min_prec, stmt=False):
        lhs = self.parse_unary(stmt)
        # a block-like expression at statement position ends the statement (Rust's rule)
        if stmt and lhs[0] in BLOCKLIKE:
            return lhs
        while True:
            tok = self.peek()
            if tok[0] != "op" or tok[1] not in BINARY:
                break
            prec = BINARY[tok[1]]
            if prec < min_prec:
                break
            # closure bars / or-patterns never appear in operator position here
            self.i += 1
            line = self.line()
            rhs = self.parse_binary(prec + 1)
            lhs = ("bin", tok[1], lhs, rhs, line)
        return lhs

    def parse_unary(self, stmt=False):
        if stmt and (self.at("if") or self.at("match") or self.at("for") or self.at("while") or self.at("loop")
                     or self.at("{")):
            return self.parse_primary()
        if self.accept("-"):
            return ("neg", self.parse_unary())
        if self.accept("!"):
            return ("not", self.parse_unary())
        if self.accept("&"):
            self.accept("mut")
            return self.parse_unary()              # references are transparent
        if self.at("&&"):                          # `&&x`
            self.i += 1
            return self.parse_unary()
        if self.accept("*"):
            return self.parse_unary()              # so are dereferences
        e = self.parse_postfix(self.parse_primary())
        while self.at("as"):
            self.i += 1
            ty = self.parse_type()
            e = ("cast", e, ty[1] if ty[0] == "path" else "?")
        return e

    def parse_args(self, close=")"):
        args = []
        while not self.accept(close):
            args.append(self.parse_expr())
            if not self.at(close):
                self.expect(",")
        return args

    def parse_postfix(self, e):
        while True:
            line = self.line()
            if self.accept("?"):
                e = ("try", e, line)
            elif self.at(".") :
                self.i += 1
                tok = self.peek()
                if tok[0] == "num":                # tuple field
                    self.i += 1
                    e = ("tfield", e, int(tok[1]))
                    continue
                name = self.ident()
                if self.at("::"):                  # method turbofish  .collect::<Vec<f64>>()
                    self.i += 1
                    self.parse_generic_args()
                if self.accept("("):
                    e = ("method", e, name, self.parse_args(), line)
                else:
                    e = ("field", e, name, line)
            elif self.accept("("):
                e = ("call", e, self.parse_args(), line)
            elif self.accept("["):
                idx = self.parse_expr()
                self.expect("]")
                e = ("index", e, idx, line)
            else:
                return e

    @staticmethod
    def number(text):
        t = text.replace("_", "")
        for suf in INT_SUFFIX:
            if t.endswith(suf):
                return int(t[:-len(suf)])
        if t.endswith("f64") or t.endswith("f32"):
            return float(t[:-3])
        if "." in t or "e" in t or "E" in t:
            return float(t)
        return int(t)

    def parse_primary(self):
        tok = self.peek()
        line = self.line()
        if tok[0] == "num":
            self.i += 1
            return ("lit", self.number(tok[1]))
        if tok[0] == "str":
            self.i += 1
            return ("lit", bytes(tok[1][1:-1], "utf-8").decode("unicode_escape"))
        if self.accept("("):
            if self.accept(")"):
                return ("tuple", [])
            first = self.parse_expr()
            if self.accept(")"):
                return ("paren", first)
            parts = [first]
            while not self.accept(")"):
                self.expect(",")
                if self.at(")"):
                    continue
                parts.append(self.parse_expr())
            return ("tuple", parts)
        if self.accept("["):
            if self.accept("]"):
                return ("array", [])
            first = self.parse_expr()
            if self.accept(";"):
                count = self.parse_expr()
                self.expect("]")
                return ("repeat", first, count)
            parts = [first]
            while not self.accept("]"):
                self.expect(",")
                if self.at("]"):
                    continue
                parts.append(self.parse_expr())
            return ("array", parts)
        if self.at("{"):
            return self.parse_block()
        if self.at("|") or self.at("||"):
            params = []
            if self.accept("||"):
                pass
            else:
                self.expect("|")
                while not self.accept("|"):
                    pat = self.parse_pattern()
                    if self.accept(":"):
                        self.parse_type()
                    params.append(pat)
                    self.accept(",")
            body = self.parse_expr()
            return ("closure", params, body)
        if tok[0] != "id":
            raise RustSyntaxError(f"{self.name}:{line}: unexpected token {tok[1]!r}")
        kw = tok[1]
        if kw == "if":
            return self.parse_if()
        if kw == "match":
            self.i += 1
            scrut = self.parse_expr()
            self.expect("{")
            arms = []
            while not self.accept("}"):
                pats = [self.parse_pattern()]
                while self.accept("|"):
                    pats.append(self.parse_pattern())
                guard = None
                if self.accept("if"):
                    guard = self.parse_expr()
                self.expect("=>")
                body = self.parse_expr()
                self.accept(",")
                arms.append((pats, guard, body))
            return ("match", scrut, arms, line)
        if kw == "for":
            self.i += 1
            pat = self.parse_pattern()
            self.expect("in")
            it = self.parse_expr()
            body = self.parse_block()
            return ("for", pat, it, body, line)
        if kw == "while":
            self.i += 1
            if self.accept("let"):
                pat = self.parse_pattern()
                self.expect("=")
                e = self.parse_expr()
                body = self.parse_block()
                return ("whilelet", pat, e, body, line)
            cond = self.parse_expr()
            body = self.parse_block()
            return ("while", cond, body, line)
        if kw == "loop":
            self.i += 1
            return ("loop", self.parse_block(), line)
        if kw == "return":
            self.i += 1
            if self.at(";") or self.at("}"):
                return ("return", None)
            return ("return", self.parse_expr())
        if kw == "break":
            self.i += 1
            return ("break",)
        if kw == "continue":
            self.i += 1
            return ("continue",)
        if kw in ("true", "false"):
            self.i += 1
            return ("lit", kw == "true")
        # path:  a::b::<T>::c   |  macro:  name!(...) / name![...]
        segs = [self.ident()]
        while self.at("::"):
            self.i += 1
            if self.at("<"):
                self.parse_generic_args()
                continue
            segs.append(self.ident())
        if self.at("!") and (self.at("(", 1) or self.at("[", 1)):
            self.i += 1
            close = ")" if self.peek()[1] == "(" else "]"
            self.i += 1
            if segs[-1] == "vec":
                if self.accept(close):
                    return ("array", [])
                first = self.parse_expr()
                if self.accept(";"):
                    count = self.parse_expr()
                    self.expect(close)
                    return ("repeat", first, count)
                parts = [first]
                while not self.accept(close):
                    self.expect(",")
                    if self.at(close):
                        continue
                    parts.append(self.parse_expr())
                return ("array", parts)
            return ("macro", segs[-1], self.parse_args(close), line)
        if len(segs) == 1:
            return ("var", segs[0], line)
        return ("path", "::".join(segs), line)

    def parse_if(self):
        line = self.line()
        self.expect("if")
        if self.accept("let"):
            pat = self.parse_pattern()
            self.expect("=")
            e = self.parse_expr()
            then = self.parse_block()
            other = self.parse_else()
            return ("iflet", pat, e, then, other, line)
        cond = self.parse_expr()
        then = self.parse_block()
        other = self.parse_else()
        return ("if", cond, then, other, line)

    def parse_else(self):
        if not self.accept("else"):
            return None
        if self.at("if"):
            return self.parse_if()
        return self.parse_block()


def parse_rust(text: str, name: str = "<rust>"):
    return Parser(text, name).parse_file()
