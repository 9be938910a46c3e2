"""LIKE oracle — TEST INFRASTRUCTURE ONLY (never imported by the product path).

The reference has no LIKE (sqlparser 0.6 parses `s LIKE 'p'` and `s NOT LIKE 'p'`, plan_parser.rs refuses every operator it
does not map), so there is no reference behaviour to restate: this file STATES the semantics the device operator implements
and tests/test_like_host.py cross-checks it against pyarrow's `match_like`.  parity unpinned by the reference.

  * `%` matches any sequence of zero or more characters, newlines included;
  * `_` matches exactly one character, i.e. one UTF-8 code point (1 to 4 bytes);
  * `\\` makes the next pattern character literal (`\\%`, `\\_`, `\\\\`); a pattern that ends in an unpaired `\\` is an error
    (pyarrow drops that backslash instead: the one deliberate difference);
  * every other character matches itself: case-sensitive, bytewise, NUL and newline included;
  * a NULL string gives NULL for LIKE and for NOT LIKE.
"""
from __future__ import annotations

import re
from typing import Optional, Sequence, Union

TRAILING_ESCAPE = "LIKE pattern ends with the escape character \\"


def like_regex(pattern: Union[str, bytes]) -> "re.Pattern":
    """the pattern as an anchored-by-fullmatch regular expression over code points"""
    p = pattern.decode() if isinstance(pattern, bytes) else pattern
    out, i = [], 0
    while i < len(p):
        c = p[i]
        if c == "\\":
            if i + 1 == len(p):
                raise ValueError(TRAILING_ESCAPE)
            out.append(re.escape(p[i + 1]))
            i += 2
            continue
        out.append(".*" if c == "%" else "." if c == "_" else re.escape(c))
        i += 1
    return re.compile("".join(out), re.DOTALL)


def match_like(value: Optional[Union[str, bytes]], pattern: Union[str, bytes], negate: bool = False) -> Optional[bool]:
    if value is None:
        return None
    v = value.decode() if isinstance(value, bytes) else value
    return (like_regex(pattern).fullmatch(v) is not None) != negate


def like_bits(values: Sequence[Optional[Union[str, bytes]]], pattern: Union[str, bytes], negate: bool = False) -> list:
    """what fq_utf8_like writes, one bool per row: the match, negated by `negate`, and False for a NULL row"""
    rx = like_regex(pattern)
    return [False if v is None else (rx.fullmatch(v.decode() if isinstance(v, bytes) else v) is not None) != negate for v in values]
