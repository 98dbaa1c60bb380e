"""Generates tests/golden/swift_reference.json: what tests/test_swift_patches.py needs to know about the upstream Wax
files that swift/patches/*.patch apply to -- line counts, SHA-256 digests and needle counts, never their text.

    python tests/golden/make_swift_reference.py <upstream Wax checkout>

Run it again whenever the patches are regenerated (swift/patches/make_patches.py) against a new upstream revision.
"""
import json
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from helpers import GOLDEN, SWIFT_RECORD, swift_reference_record  # noqa: E402


def main():
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    path = GOLDEN / SWIFT_RECORD
    path.write_text(json.dumps(swift_reference_record(Path(sys.argv[1])), indent=1) + "\n")
    print(path, path.stat().st_size, "bytes")


if __name__ == "__main__":
    main()
