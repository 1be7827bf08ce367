"""Public surface inherited from the reference's pipeline classes (SURVEY.md 8b): CPU-checkable parts."""
import os

import numpy as np

PINS = os.path.join(os.path.dirname(__file__), "golden", "reference_pins.npz")


def test_receptive_field_matches_reference_helpers():
    """(size, step, center) the reference's receptive_field helpers give for the WavLM conv stack (reference_pins.npz)."""
    from diarizen_b200.segmentation import SegmentationModel
    size, step, center = np.load(PINS)["receptive_field"]
    sw = SegmentationModel._receptive_field.fget(None)
    assert (sw.start, sw.duration, sw.step) == ((center - (size - 1) / 2) / 16000, size / 16000, step / 16000)


def test_annotation_drops_empty_segments_and_orders_tracks():
    from diarizen_b200.annotation import Annotation, Segment
    a = Annotation(uri="u")
    a[Segment(1.0, 1.0), 0] = 0           # a turn made of a single frame: empty, dropped (pyannote.core semantics)
    a[Segment(0.5, 2.0), 10] = 10
    a[Segment(0.5, 2.0), 2] = 2
    a[Segment(0.25, 0.75), 1] = 1
    got = [(s.start, s.end, l) for s, _, l in a.itertracks(yield_label=True)]
    assert got == [(0.25, 0.75, 1), (0.5, 2.0, 10), (0.5, 2.0, 2)]        # tracks of one segment in str order: "10" < "2"
    assert a.to_rttm().splitlines()[0] == "SPEAKER u 1 0.250 0.500 <NA> <NA> 1 <NA> <NA>"


def test_to_annotation_matches_reference_binarize():
    """pipeline.to_annotation on a {0,1} matrix (runs of frames, and a zero-length turn on the last frame) == the RTTM of the
    reference's Binarize on the same matrix (reference_pins.npz, produced through oracle/ref_glue.py)."""
    from diarizen_b200.pipeline import DiariZenPipeline
    z = np.load(PINS)
    assert DiariZenPipeline.to_annotation(z["binarize/disc"], "x").to_rttm() == str(z["binarize/rttm"])
