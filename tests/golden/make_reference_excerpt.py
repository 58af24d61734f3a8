"""Writes tests/golden/reference_excerpt/: the 23 files of the reference crate (jalberse/RayTracingInOneWeekendInRust)
that rust/shimmer-patch/shimmer-b200.patch changes, as far as the repository records them.

Each file keeps, at its original line numbers, the lines the patch shows of it (context and removed lines) and the
reference text each edit of make_patch.py names; every other line is a numbered placeholder comment.
tests/test_rust_binding.py applies the patch to this copy and checks that make_patch.py, run against it, writes the
committed patch byte for byte.  The excerpt pins the patch as it is when this script runs: run it again only after
regenerating the patch from a full checkout of the reference crate.

    python tests/golden/make_reference_excerpt.py
"""
import re
import shutil
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[2]
PATCH = ROOT / "rust" / "shimmer-patch" / "shimmer-b200.patch"
OUT = Path(__file__).resolve().parent / "reference_excerpt"
sys.path.insert(0, str(ROOT / "rust" / "shimmer-patch"))
import make_patch  # noqa: E402


def shown_lines(patch_text):
    """{path: [line text, or None where the patch does not show it]} of the pre-image of each file the patch changes."""
    files, path, lines = {}, None, patch_text.split("\n")
    i = 0
    while i < len(lines):
        line = lines[i]
        if line.startswith("+++ b/"):
            path = line[len("+++ b/"):]
        elif line.startswith("@@"):
            m = re.match(r"@@ -(\d+)(?:,(\d+))? \+\d+(?:,(\d+))? @@", line)
            start, n_old, n_new = int(m.group(1)), int(m.group(2) or 1), int(m.group(3) or 1)
            seen_old = seen_new = 0
            while seen_old < n_old or seen_new < n_new:
                i += 1
                b = lines[i]
                if b.startswith("\\"):       # "\ No newline at end of file"
                    continue
                if b[:1] in (" ", "-"):
                    known = files.setdefault(path, [])
                    n = start + seen_old           # 1-based
                    known.extend([None] * (n - len(known)))
                    known[n - 1] = b[1:]
                    seen_old += 1
                seen_new += b[:1] in (" ", "+")
        i += 1
    return files


def place(known, old):
    """Writes the reference text ``old`` (whole lines, the last one possibly a prefix) into ``known`` where it agrees
    with the most shown lines; a prefix is kept as a prefix, the rest of its line marked unknown."""
    parts = old.split("\n")
    whole, prefix = parts[:-1], parts[-1]
    want = whole + ([prefix] if prefix else [])

    def fits(p):
        score = 0
        for k, part in enumerate(want):
            have = known[p + k] if p + k < len(known) else None
            if have is None:
                continue
            if not (have == part if k < len(whole) else have.startswith(part)):
                return -1
            score += 1
        return score

    scores = {p: fits(p) for p in range(len(known))}
    best = max(scores.values())
    at = [p for p, s in scores.items() if s == best]
    assert best > 0 and len(at) == 1, f"cannot place {old!r}"
    p = at[0]
    known.extend([None] * (p + len(want) - len(known)))
    for k, part in enumerate(want):
        if known[p + k] is None:
            known[p + k] = part if k < len(whole) else part + f" // rest of line {p + k + 1}: not recorded"


def main():
    files = shown_lines(PATCH.read_text())
    for path, edits in make_patch.EDITS.items():
        for old, _ in edits:
            place(files[path], old)
    shutil.rmtree(OUT, ignore_errors=True)
    for path, known in files.items():
        comment = "#" if path.endswith(".toml") else "//"
        text = "".join((line if line is not None else f"{comment} line {n}: not recorded") + "\n"
                       for n, line in enumerate(known, 1))
        (OUT / path).parent.mkdir(parents=True, exist_ok=True)
        (OUT / path).write_text(text)
        print(path, f"{sum(line is not None for line in known)} of {len(known)} lines recorded")


if __name__ == "__main__":
    main()
