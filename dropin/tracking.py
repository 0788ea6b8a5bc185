"""Drop-in for the reference's ``tracking`` module (reference ``initialize.py:458``, ``:502``)."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from softgnss_python_b200.tracking import TrackingResult, cno_vsm, tracking  # noqa: E402,F401
