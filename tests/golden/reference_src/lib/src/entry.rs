    /// ```
    #[inline]
    pub fn reader(&self, option: impl ReadOption) -> io::Result<EntryDataReader<'_>> {
        let decrypt_reader = decrypt_reader(
            self.encoded_reader(),
            self.header.encryption,
            &self.header.to_bytes(),
        )?;
        let reader = decompress_reader(decrypt_reader, self.header.compression)?;
        Ok(EntryDataReader(EntryReader(reader)))
    }
}

