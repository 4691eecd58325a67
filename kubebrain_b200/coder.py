"""Host-side mirror of the reference's internal key codec (pkg/backend/coder/normal.go:25-70, rev.go:22-47).

Only used to build range bounds and to read results; the per-record decode of a scan runs on the GPU
(the decoded columns of the record directory, csrc/kb_decode.cuh).
"""
from __future__ import annotations

import struct
from typing import Tuple

MAGIC = b"\x57\xfb\x80\x8b"  # normal.go:26
SPLIT = 0x24  # '$' normal.go:31

REVISION_VALUE_LENGTH = 8  # rev.go:23
REVISION_VALUE_LENGTH_WITH_DELETION_FLAG = 9  # rev.go:24


class DecodeError(ValueError):
    pass


class ErrInvalidRevFormat(ValueError):  # rev.go:28
    pass


class NormalCoder:
    """coder.Coder (pkg/backend/coder/interface.go:18-28)"""

    def encode_object_key(self, user_key: bytes, revision: int) -> bytes:  # normal.go:42-50
        return MAGIC + user_key + b"$" + struct.pack(">Q", revision)

    def encode_revision_key(self, user_key: bytes) -> bytes:  # normal.go:53-55
        return self.encode_object_key(user_key, 0)

    def decode(self, internal_key: bytes) -> Tuple[bytes, int]:  # normal.go:58-70
        if len(internal_key) < 13:
            # the Go code indexes without a length check and would panic; the mirror raises
            raise DecodeError("internal key shorter than 13 bytes: %s" % internal_key.hex())
        if internal_key[:4] != MAGIC:
            raise DecodeError("magic number not right for object key %s" % internal_key.hex())
        if internal_key[-9] != SPLIT:
            raise DecodeError("split byte not right for object key %s" % internal_key.hex())
        return internal_key[4:-9], struct.unpack(">Q", internal_key[-8:])[0]


def parse_revision(revision_bytes: bytes) -> Tuple[int, bool]:  # rev.go:32-47
    if len(revision_bytes) == REVISION_VALUE_LENGTH:
        return struct.unpack(">Q", revision_bytes)[0], False
    if len(revision_bytes) == REVISION_VALUE_LENGTH_WITH_DELETION_FLAG:
        return struct.unpack(">Q", revision_bytes[:8])[0], True
    raise ErrInvalidRevFormat("invalid format of revision bytes")


def prefix_end(prefix: bytes) -> bytes:
    """pkg/backend/util.go:70-83"""
    end = bytearray(prefix)
    for i in range(len(end) - 1, -1, -1):
        if end[i] < 0xFF:
            end[i] += 1
            return bytes(end[: i + 1])
    return b"\x00"  # noPrefixEnd
