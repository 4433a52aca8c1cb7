import json
import os
from pathlib import Path


def reference_dir() -> Path:
    """Checkout of the original RoboCupVision project: $RCV_REFERENCE_DIR, else BASELINE.json's reference_path."""
    if os.environ.get("RCV_REFERENCE_DIR"):
        return Path(os.environ["RCV_REFERENCE_DIR"])
    return Path(json.loads((Path(__file__).resolve().parent.parent / "BASELINE.json").read_text())["reference_path"])
