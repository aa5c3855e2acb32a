/*
 * bamerr.h — messages of a rejected BAM region, shared by the host decoder (bamdec.c) and the device decoder
 * (bamgpu.cuh, formatted by himut_b200.cu), so that both reject the same input with the same text.
 * Every format takes a string (the BAM path or the record's query name, see REC_ERR_ON_PATH) and a long.
 */
#ifndef HIMUT_BAMERR_H
#define HIMUT_BAMERR_H

enum {
  E_CS_TOKEN = 1, E_CS_PAST, E_N_MATCH, E_CS_LONG, E_SUB_N, E_SPAN_REF, E_SPAN_QRY, /* cs -> ops (record decode) */
  E_MD_TOKEN, E_MD_SPAN, E_CIGAR_OP,         /* CIGAR + MD:Z -> ops (record decode, records without cs:Z) */
  E_BLOCK_SIZE, E_FIELDS, E_TAG_UNTERM, E_TAG_B, E_TAG_TYPE, E_TAG_PAST, E_NO_CS, E_NO_QUAL, /* record selection */
  E_TRUNC_REC,                               /* a record runs past the end of the data */
  E_INFLATE, E_CRC, E_BAI_ENTRY,             /* device decoder only: BGZF block / index problems */
  E_N_CODES
};
static const char* const REC_ERR[E_N_CODES] = {
    "", "%s: unsupported cs token (%ld)", "%s: cs runs past the read (%ld)",
    "%s: read base outside A/C/G/T under a cs match (reference: KeyError) (%ld)",
    "%s: cs long-form bases disagree with SEQ at query %ld",
    "%s: substitution to a base outside A/C/G/T (the reference pileup raises KeyError) (%ld)",
    "%s: cs reference span != CIGAR span (%ld)", "%s: cs query span != aligned query span (%ld)",
    "%s: unsupported MD:Z token (%ld)", "%s: MD:Z and CIGAR disagree at reference offset %ld",
    "%s: unsupported CIGAR op (N, P, or a clip inside the alignment) at CIGAR index %ld",
    "malformed BAM record in %s: block_size %ld", "malformed BAM record in %s: fields run past block_size %ld",
    "malformed BAM record %s: unterminated %ld tag", "malformed BAM record %s: truncated B tag (%ld)",
    "unknown tag type in record %s (%ld)", "malformed BAM record %s: a tag runs past the record (%ld)",
    "%s has no cs:Z tag (the reference raises KeyError in BAM.__init__) (%ld)", "%s has no base qualities (%ld)",
    "truncated BAM record in %s (%ld)",
    "BGZF block of %s does not inflate to its ISIZE (block %ld)", "BGZF block of %s fails its CRC32 (block %ld)",
    "BAI does not point at record starts in %s (entry %ld)"};
/* the codes whose %s is the BAM path; the others take the record's query name */
#define REC_ERR_ON_PATH(code) ((code) == E_BLOCK_SIZE || (code) == E_FIELDS || (code) >= E_TRUNC_REC)

#endif
