"""Where the checkout of the original project (ajbrock/Neural-Photo-Editor) is, whose own files the fixture generators
under tests/golden execute: $NPE_REFERENCE, else the `reference_path` that BASELINE.json records."""
import json
import os

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def reference_dir():
    """the checkout's directory, or None where there is none (its sources are not part of this repository)"""
    with open(os.path.join(ROOT, "BASELINE.json")) as f:
        path = os.environ.get("NPE_REFERENCE") or json.load(f)["reference_path"]
    return path if os.path.isdir(path) else None
