"""Shared test helpers: a list-based model of the engine's mutation semantics, comparators."""
from __future__ import annotations

import json
from pathlib import Path

import numpy as np

GOLDEN = Path(__file__).resolve().parent / "golden"


class EngineModel:
    """Reference mutation semantics (MetalVectorEngine.swift:330-444) on plain Python lists:
    upsert by frameId (overwrite in place, else append), order-preserving remove, no-op for unknown ids.
    Search goes through the oracle."""

    def __init__(self, oracle, metric: int, dims: int):
        self.o, self.metric, self.dims = oracle, metric, dims
        self.ids: list[int] = []
        self.rows: list[np.ndarray] = []

    def add(self, frame_id, vector):
        v = np.asarray(vector, np.float32)
        assert v.size == self.dims
        if frame_id in self.ids:
            self.rows[self.ids.index(frame_id)] = v
        else:
            self.ids.append(frame_id)
            self.rows.append(v)

    def add_batch(self, frame_ids, vectors):
        for i, v in zip(frame_ids, vectors):
            self.add(i, v)

    def remove(self, frame_id):
        if frame_id in self.ids:
            idx = self.ids.index(frame_id)
            del self.ids[idx]
            del self.rows[idx]

    def corpus(self):
        return np.stack(self.rows).astype(np.float32) if self.rows else np.zeros((0, self.dims), np.float32)

    def search(self, query, top_k, mode=None):
        mode = self.o.ACC_F32_TREE if mode is None else mode
        if not self.rows:
            return []
        rows, d, s = self.o.search(self.metric, self.corpus(), query, top_k, mode=mode)
        return [(self.ids[int(r)], float(sc)) for r, sc in zip(rows, s)]


def assert_tie_aware_order(got_ids, ref_ids, ref_scores_f64, tol):
    """ids must match position by position, except inside groups whose fp64-oracle scores are within `tol`
    of each other (where fp32 rounding order may legitimately permute neighbours)."""
    got_ids, ref_ids = list(got_ids), list(ref_ids)
    assert len(got_ids) == len(ref_ids)
    i = 0
    n = len(ref_ids)
    while i < n:
        j = i
        while j + 1 < n and abs(ref_scores_f64[j + 1] - ref_scores_f64[j]) <= tol:
            j += 1
        # positions i..j form a near-tie group; the last group may also trade members with rank n+1.. if the
        # boundary is a near tie -- callers pass one extra reference row to detect that.
        assert sorted(got_ids[i:j + 1]) == sorted(ref_ids[i:j + 1]) or j == n - 1, (
            f"order differs outside a near-tie at ranks {i}..{j}: got {got_ids[i:j + 1]} ref {ref_ids[i:j + 1]}")
        i = j + 1


def load_json(name):
    return json.loads((GOLDEN / name).read_text())


# -- the Swift patches (swift/patches/*.patch) against a record of the upstream files they apply to
SWIFT_PATCHES = Path(__file__).resolve().parents[1] / "swift" / "patches"
SWIFT_RECORD = "swift_reference.json"
# the switch arms and enum cases the patch generator rewrites, counted over each whole upstream file
SWIFT_NEEDLES = ("case .metal(let engine):", "case .cuda(let engine):", "case metal(MetalVectorEngine)",
                 "case cuda(CUDAVectorEngine)")


def parse_patch(text: str):
    """A unified diff of one file -> (path, hunks); a hunk is (old_start, old_len, new_start, new_len, [(tag, line)])
    with tag one of ' ', '-', '+' and each line carrying its newline."""
    import re
    rel, hunks = None, []
    for line in text.splitlines(True):
        if line.startswith("--- a/"):
            rel = line[6:].strip()
        elif line.startswith("+++ "):
            continue
        elif line.startswith("@@"):
            m = re.match(r"@@ -(\d+)(?:,(\d+))? \+(\d+)(?:,(\d+))? @@", line)
            hunks.append((int(m[1]), int(m[2] or 1), int(m[3]), int(m[4] or 1), []))
        elif hunks and line[:1] in (" ", "-", "+"):
            hunks[-1][4].append((line[0], line[1:]))
        else:
            raise ValueError(f"unexpected line in a patch: {line!r}")
    return rel, hunks


def hunk_pre_image(hunk) -> str:
    return "".join(l for tag, l in hunk[4] if tag in " -")


def sha256_text(text: str) -> str:
    import hashlib
    return hashlib.sha256(text.encode("utf-8")).hexdigest()


def generator_blocks() -> list:
    """The upstream blocks make_patches.py rewrites verbatim: the plain-string `old` arguments of its must_replace()."""
    import ast
    tree = ast.parse((SWIFT_PATCHES / "make_patches.py").read_text())
    return [n.args[1].value for n in ast.walk(tree)
            if isinstance(n, ast.Call) and getattr(n.func, "id", None) == "must_replace"
            and isinstance(n.args[1], ast.Constant) and isinstance(n.args[1].value, str)]


def swift_reference_record(ref_root: Path) -> dict:
    """What the Swift-patch tests need to know about the upstream files, without their text: each file's line count,
    digest and needle counts, the digest of the upstream lines every hunk replaces, and where each block the generator
    rewrites starts (its text is in make_patches.py)."""
    files = {}
    for patch in sorted(SWIFT_PATCHES.glob("*.patch")):
        rel, hunks = parse_patch(patch.read_text())
        text = (Path(ref_root) / rel).read_text()
        lines = text.splitlines(True)
        blocks = []
        for block in generator_blocks():
            if text.count(block) == 1:
                start = text[:text.index(block)].count("\n") + 1
                blocks.append({"start": start, "lines": block.count("\n"), "sha256": sha256_text(block)})
        files[rel] = {
            "lines": len(lines), "trailing_newline": text.endswith("\n"), "sha256": sha256_text(text),
            "counts": {n: text.count(n) for n in SWIFT_NEEDLES},
            "hunks": [{"old_start": h[0], "old_len": h[1], "sha256": sha256_text("".join(lines[h[0] - 1:h[0] - 1 + h[1]]))}
                      for h in hunks],
            "generator_blocks": sorted(blocks, key=lambda b: b["start"]),
        }
        # how often each line of the hunks and blocks occurs upstream: difflib treats frequent lines as junk when it
        # aligns a diff, so the stand-in repeats them as often as the upstream file does
        known = set(hunk_pre_image(h) for h in hunks) | {b for b in generator_blocks() if text.count(b) == 1}
        known_lines = {l for chunk in known for l in chunk.splitlines(True)}
        files[rel]["line_counts"] = {sha256_text(l): lines.count(l) for l in sorted(known_lines)}
    return {"_comment": "upstream Wax files the Swift patches apply to: line counts, positions and SHA-256 digests "
                        "only (tests/golden/make_swift_reference.py)", "files": files}


def swift_reference_skeleton(rel: str, hunks, record: dict) -> str:
    """A stand-in for an upstream file: the blocks the generator rewrites and the lines the patch's hunks name (their
    pre-images) at their recorded positions, a distinct placeholder line everywhere else."""
    n = record["lines"]
    lines = [f"// upstream line {i + 1}, untouched by the patch\n" for i in range(n)]
    by_digest = {sha256_text(b): b for b in generator_blocks()}
    for b in record["generator_blocks"]:
        assert b["sha256"] in by_digest, (rel, b)      # make_patches.py still rewrites this upstream block
        lines[b["start"] - 1:b["start"] - 1 + b["lines"]] = by_digest[b["sha256"]].splitlines(True)
    for h in hunks:
        assert 1 <= h[0] and h[0] - 1 + h[1] <= n, (rel, h[:4])
        lines[h[0] - 1:h[0] - 1 + h[1]] = hunk_pre_image(h).splitlines(True)
    assert len(lines) == n, rel
    # repeat known lines in placeholder slots, farthest from any recorded line first, until each occurs as often as
    # upstream
    placed = [i for i, l in enumerate(lines) if not l.startswith("// upstream line ")]
    free = sorted((i for i, l in enumerate(lines) if l.startswith("// upstream line ")),
                  key=lambda i: (min(abs(i - j) for j in placed), i))
    for line in sorted(set(lines) - set(lines[i] for i in free)):
        for _ in range(record["line_counts"][sha256_text(line)] - lines.count(line)):
            lines[free.pop()] = line
    text = "".join(lines)
    return text if record["trailing_newline"] else text[:-1]
