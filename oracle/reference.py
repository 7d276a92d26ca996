"""Where the original project's sources are, for the tests and the benchmark arm that run its code unchanged."""
import os


def reference_dir():
    """A checkout of the original project (CoderLinxin/Single-Image-Super-Resolution-Application) named by HITSIR_REFERENCE_DIR, or
    None.  It is not part of this repository; what needs it skips (tests) or says it ran without it (bench.py)."""
    root = os.environ.get("HITSIR_REFERENCE_DIR")
    if root and os.path.exists(os.path.join(root, "models", "hit_sir_pro.py")):
        return root
    return None
