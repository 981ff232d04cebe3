#!/usr/bin/env python
"""Launch LibKGE's own command line (`kge start|resume|eval|...`, kge/cli.py) with the kge_b200 plugin importable:

    python scripts/kge_cli.py start my-job.yaml --job.device cuda

Locates the reference (installed LibKGE, $KGE_REFERENCE_ROOT or oracle/_ref — oracle/install_ref.py), stubs the
optional third-party modules it imports at module level but does not use for training / evaluation, puts this
repository on sys.path (so `modules: [..., kge_b200.plugin]` resolves) and hands over to kge.cli.main().  Nothing of
LibKGE is modified."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from kge_b200 import hostenv  # noqa: E402

hostenv.import_kge()
from kge.cli import main  # noqa: E402

if __name__ == "__main__":
    main()
