"""Host-side reader of the index image written by bbq_index_save (csrc/bbq_io.cuh): <prefix>.vemb + <prefix>.veb.

The field names are the reference's MetadataFormat / VectorDataFormat (src/types.ts:78-113) and the file extensions
its FILE_EXTENSIONS (src/constants.ts:52-57).  Pure file parsing for tools and tests — nothing here scores or
quantises, and the search path never goes through it (bbq_index_load streams the file into HBM natively).
"""
from __future__ import annotations

import struct

import numpy as np

MAGIC = b"BVECb200"
VERSION = 1
SECTION_ALIGN = 4096
# char magic[8]; u32 version, fieldNumber, vectorEncodingOrdinal, vectorSimilarityOrdinal, dimensions, indexBits,
# rowBytes, reserved; u64 vectorCount, vectorDataOffset, vectorDataLength, lower/upper/additional/componentSum offsets;
# f64 centroidSquareMagnitude; u64 checksum[5]
_HEADER = struct.Struct("<8s8I7Qd5Q")
HEADER_BYTES = _HEADER.size
SECTIONS = ("binaryValues", "lowerInterval", "upperInterval", "additionalCorrection", "quantizedComponentSum")
SIMILARITY_ORDINALS = ("EUCLIDEAN", "COSINE", "MAXIMUM_INNER_PRODUCT")


class ImageFormatError(ValueError):
    pass


def row_bytes_for(dimensions: int) -> int:
    return ((dimensions + 7) // 8 + 15) // 16 * 16


def section_layout(vector_count: int, dimensions: int):
    """[(name, offset, bytes)] of the five .veb sections."""
    sizes = (vector_count * row_bytes_for(dimensions), vector_count * 8, vector_count * 8, vector_count * 8,
             vector_count * 4)
    out, off = [], 0
    for name, size in zip(SECTIONS, sizes):
        out.append((name, off, size))
        off = (off + size + SECTION_ALIGN - 1) // SECTION_ALIGN * SECTION_ALIGN
    return out


def section_checksum(raw, first_word: int = 0) -> int:
    """sum over 32-bit words of splitmix64(index << 32 | word), mod 2^64 — what k_section_checksum computes.
    first_word: the position of raw's first word in its section (rows [r, ...) of a section of stride S bytes start at
    word r * S / 4), so the checksums of the slices of a section add up, mod 2^64, to the checksum of the section."""
    words = np.frombuffer(memoryview(raw), dtype="<u4").astype(np.uint64)
    total = 0
    step = 1 << 22
    with np.errstate(over="ignore"):
        for s in range(0, words.size, step):
            w = words[s:s + step]
            z = (np.arange(first_word + s, first_word + s + w.size, dtype=np.uint64) << np.uint64(32)) | w
            z = z + np.uint64(0x9E3779B97F4A7C15)
            z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
            z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
            z = z ^ (z >> np.uint64(31))
            total = (total + int(z.sum(dtype=np.uint64))) & 0xFFFFFFFFFFFFFFFF
    return total


def read_metadata(prefix: str) -> dict:
    """MetadataFormat (src/types.ts:95-113) of <prefix>.vemb, plus the layout fields this format adds."""
    with open(prefix + ".vemb", "rb") as f:
        blob = f.read()
    if len(blob) < HEADER_BYTES:
        raise ImageFormatError("truncated metadata file")
    (magic, version, field_number, encoding, similarity, dimensions, index_bits, row_bytes, _reserved, count,
     data_offset, data_length, lower_off, upper_off, add_off, sum_off, cdp, *checksums) = _HEADER.unpack_from(blob)
    if magic != MAGIC:
        raise ImageFormatError("not a BVEC metadata file")
    if version != VERSION:
        raise ImageFormatError(f"unsupported index image version {version}")
    if len(blob) != HEADER_BYTES + 4 * dimensions:
        raise ImageFormatError("metadata length does not match the dimension")
    return {
        "fieldNumber": field_number, "vectorEncodingOrdinal": encoding, "vectorSimilarityOrdinal": similarity,
        "dimensions": dimensions, "vectorDataOffset": data_offset, "vectorDataLength": data_length,
        "vectorCount": count, "centroid": np.frombuffer(blob, "<f4", dimensions, HEADER_BYTES).copy(),
        "centroidSquareMagnitude": cdp,
        # additions
        "indexBits": index_bits, "rowBytes": row_bytes,
        "sectionOffsets": dict(zip(SECTIONS, (data_offset, lower_off, upper_off, add_off, sum_off))),
        "sectionChecksums": dict(zip(SECTIONS, checksums)),
        "similarityFunction": SIMILARITY_ORDINALS[similarity] if similarity < 3 else None,
    }


def read_vector_data(prefix: str, meta: dict | None = None, verify: bool = True) -> dict:
    """The VectorDataFormat columns (src/types.ts:78-90) of <prefix>.veb as numpy views on a memory map;
    binaryValues is [vectorCount, ceil(dimensions/8)] (the 16-byte row padding is cut off)."""
    meta = meta or read_metadata(prefix)
    n, dim = meta["vectorCount"], meta["dimensions"]
    mm = np.memmap(prefix + ".veb", dtype=np.uint8, mode="r")
    layout = section_layout(n, dim)
    if mm.size < layout[-1][1] + layout[-1][2]:
        raise ImageFormatError("truncated vector data file")
    out = {}
    dtypes = (np.uint8, "<f8", "<f8", "<f8", "<u4")
    for (name, off, size), dt in zip(layout, dtypes):
        if meta["sectionOffsets"][name] != off:
            raise ImageFormatError(f"unexpected offset of section {name}")
        raw = mm[off:off + size]
        if verify and section_checksum(raw) != meta["sectionChecksums"][name]:
            raise ImageFormatError(f"checksum mismatch in section {name}")
        out[name] = raw.view(dt)
    out["binaryValues"] = out["binaryValues"].reshape(n, meta["rowBytes"])[:, :(dim + 7) // 8]
    return out
