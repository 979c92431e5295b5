"""halo2_regex_b200 — B200-native (sm_100a) witness generation for zkemail/halo2-regex's DFA path.

Host mirror of the reference's `halo2_regex::{defs, RegexVerifyConfig}` over the C ABI in include/b2r.h.
Importing this package loads halo2_regex_b200/libb2r.so and fails loudly if it has not been built (no CPU fallback).
"""
from . import _abi  # noqa: F401
from ._ffi import LIB_PATH, SYMBOLS, last_error, lib  # noqa: F401
from .buffers import HostOutputs, PinnedAllocator, compare_outputs  # noqa: F401
from .defs import AllstrRegexDef, RegexDefs, RegexParseError, SubstrRegexDef  # noqa: F401
from .regex import (AssignedRegexResult, DeviceOutputs, InvalidTransitionError, RegexVerifyConfig,  # noqa: F401
                    StringMultOutputs, StringMultPacked, StringTooLongError)

from . import vrm  # noqa: F401,E402  (host-side definition compiler: regex JSON -> lookup text files)

__version__ = "0.1.0"
