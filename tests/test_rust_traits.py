"""The Rust crate (rust/) is not compiled by the test-suite, so its plugin boundary is pinned textually: the
REQUIRED items of the four strategy traits must equal the reference's token for token
(src/interp1d/strategies/mod.rs:12-65, src/interp2d/strategies/mod.rs:14-73 of jonasBoss/ndarray-interp v0.6.0),
any extra trait method must be PROVIDED (have a default body), and every item the reference's user-strategy example
implements (examples/custom_strategy.rs) must exist in the crate's trait with the signature the example writes --
i.e. the example would compile unchanged next to the crate.  The two comparisons read a checkout of the reference
named by NDI_REFERENCE and are skipped without one."""
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("NDI_REFERENCE", "")
needs_reference = pytest.mark.skipif(not (REF and os.path.isdir(REF)),
                                     reason="reference sources not present (set NDI_REFERENCE to a checkout)")

# the one documented substitution: the crate's element bound (rust/README.md)
ELEM_BOUNDS = {"Num + Debug + Send": "NdiElem", "Num + PartialOrd + NumCast + Copy + Debug + Sub + Send": "NdiElem"}


def strip_comments(text):
    text = re.sub(r"//[^\n]*", "", text)
    return re.sub(r"/\*.*?\*/", "", text, flags=re.S)


def tokens(text):
    return re.findall(r"[A-Za-z_][A-Za-z_0-9]*|'[a-z_]+|::|->|=>|[{}()\[\]<>,;:&=+*?!.#-]|\d+", text)


def brace_block(text, start):
    """text[start] == '{' -> index just past the matching '}'"""
    depth = 0
    for i in range(start, len(text)):
        if text[i] == "{":
            depth += 1
        elif text[i] == "}":
            depth -= 1
            if depth == 0:
                return i + 1
    raise ValueError("unbalanced braces")


def trait(text, name):
    """(generics + where clause, {item name: (signature tokens, has default body)}) of `pub trait name`"""
    text = strip_comments(text)
    m = re.search(r"pub trait " + name + r"\b", text)
    assert m, name
    open_brace = text.index("{", m.end())
    head = text[m.end():open_brace]
    body = text[open_brace + 1:brace_block(text, open_brace) - 1]
    items, i = {}, 0
    while i < len(body):
        m2 = re.compile(r"\b(fn|const|type)\s+(\w+)").search(body, i)
        if not m2:
            break
        j = m2.end()
        depth = 0
        while True:                                   # up to the ';' or the '{' of a default body, outside <>, ()
            ch = body[j]
            if ch in "(<[":
                depth += 1
            elif ch in ")>]" and not (ch == ">" and body[j - 1] == "-"):
                depth -= 1
            elif ch == ";" and depth == 0:
                items[m2.group(2)] = (tokens(body[m2.start():j]), False)
                j += 1
                break
            elif ch == "{" and depth == 0:
                items[m2.group(2)] = (tokens(body[m2.start():j]), True)
                j = brace_block(body, j)
                break
            j += 1
        i = j
    return tokens(head), items


def normalise(toks):
    """reference tokens with the documented element-bound substitution applied; lifetimes elided or written
    (`ArrayViewMut<Sd::Elem, ..>` vs `ArrayViewMut<'_, Sd::Elem, ..>`) are the same type"""
    s = " ".join(toks)
    for ref_bound, ours in ELEM_BOUNDS.items():
        s = s.replace(" ".join(tokens(ref_bound)), ours)
    s = s.replace("< '_ , ", "< ")
    return s.replace(", )", ")").replace(", >", ">")               # a trailing comma is layout, not signature


CASES = [
    ("src/interp1d/strategies/mod.rs", "rust/src/interp1d/mod.rs", ["Interp1DStrategyBuilder", "Interp1DStrategy"]),
    ("src/interp2d/strategies/mod.rs", "rust/src/interp2d/mod.rs", ["Interp2DStrategyBuilder", "Interp2DStrategy"]),
]


@needs_reference
@pytest.mark.parametrize("ref_file,our_file,names", CASES)
def test_required_trait_items_equal_the_reference_token_for_token(ref_file, our_file, names):
    ref_text = open(os.path.join(REF, ref_file)).read()
    our_text = open(os.path.join(ROOT, our_file)).read()
    for name in names:
        ref_head, ref_items = trait(ref_text, name)
        our_head, our_items = trait(our_text, name)
        assert normalise(our_head) == normalise(ref_head), (name, "generics / where clause")
        for item, (toks, has_body) in ref_items.items():
            assert item in our_items, f"{name}::{item} is missing"
            assert normalise(our_items[item][0]) == normalise(toks), f"{name}::{item} differs from the reference"
            assert our_items[item][1] == has_body, f"{name}::{item}: required / provided differs"
        for item, (_, has_body) in our_items.items():
            if item not in ref_items:
                assert has_body, f"{name}::{item} is new and has no default: user strategies would not compile"


@needs_reference
def test_the_reference_example_compiles_against_the_crates_traits_textually():
    """examples/custom_strategy.rs, unchanged: every item of its two `impl` blocks is an item of the crate's trait
    with the same parameter list and return type (names of bindings and path prefixes aside)"""
    ex = strip_comments(open(os.path.join(REF, "examples", "custom_strategy.rs")).read())
    ours = open(os.path.join(ROOT, "rust/src/interp1d/mod.rs")).read()

    def simplify(toks):
        s = " ".join(toks)
        s = re.sub(r"\b(ndarray|ndarray_interp) :: ", "", s)          # the example writes some paths in full
        s = re.sub(r"\bmut ", "", s)                                   # `mut target` binds the same parameter
        s = re.sub(r"\b_(\w+) :", r"\1 :", s)                          # `_x:` is the parameter `x:`
        return s.replace("< '_ , ", "< ").replace(", )", ")").replace(", >", ">")

    seen = 0
    for name in ("Interp1DStrategyBuilder", "Interp1DStrategy"):
        _, our_items = trait(ours, name)
        m = re.search(r"impl<[^>]*>\s+" + name + r"<[^>]*>\s+for\s+StepInterpolator", ex)
        assert m, name
        open_brace = ex.index("{", ex.index("where", m.end()))
        body = ex[open_brace + 1:brace_block(ex, open_brace) - 1]
        for kind, item in re.findall(r"\b(fn|const|type)\s+(\w+)", body):
            if item in ("idx",):
                continue
            assert item in our_items, f"the example implements {name}::{item}, which the crate's trait lacks"
            if kind == "fn":
                sig = re.search(r"fn\s+" + item + r".*?(?=\{)", body, flags=re.S).group(0)
                want = simplify(our_items[item][0])
                got = simplify(tokens(sig))
                got = re.sub(r" ,$", "", got)                           # `where Sx2: ..,` before the body
                assert got == want, (item, got, want)
                seen += 1
    assert seen == 2                                                   # build and interp_into
    # what the example calls on the interpolator exists with those names
    for method in ("get_index_left_of", "index_point", "interp_array", "builder", "strategy", "build"):
        assert re.search(r"pub fn " + method + r"\b", ours), method


def test_readme_names_the_element_types_the_crate_instantiates():
    readme = open(os.path.join(ROOT, "rust", "README.md")).read()
    elem = open(os.path.join(ROOT, "rust", "src", "elem.rs")).read()
    for t in ("f32", "f64", "i32", "i64"):
        assert re.search(r"impl NdiElem for " + t, elem), t
        assert f"`{t}`" in readme, t
