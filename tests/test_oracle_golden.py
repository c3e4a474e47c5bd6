"""Pins both oracles (the C restatement and the compiled reference) to the reference's
own known-answer vectors (tests/golden_cases.py)."""
import pytest

import golden_cases


@pytest.mark.parametrize("case", golden_cases.ALL, ids=lambda f: f.__name__)
def test_port_golden(port, case):
    case(port)


@pytest.mark.parametrize("case", golden_cases.ALL, ids=lambda f: f.__name__)
def test_reference_golden(compiled_reference, case):
    case(compiled_reference)
