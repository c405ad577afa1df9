/// Calculates the CRC-32 checksum of a chunk type and data field.
#[inline]
pub(crate) fn chunk_crc(ty: &[u8; 4], data: &[u8]) -> u32 {
    let mut crc = crc32fast::Hasher::new();
    crc.update(ty);
    crc.update(data);
    crc.finalize()
}

/// Validates a stored chunk CRC-32 checksum.
