/* undexta -- .dexta -> .fasta.
 * Same command line, flags and file format as the reference's undexta (undexta.c:18-93); the
 * work is done by libdexb200.so on the GPU (see dxcli.h). */
#include "dxcli.h"

static int run(dx_ctx *ctx, const dx_opts *o, const uint8_t *d_in, size_t n,
               uint8_t **d_out, size_t *out_len)
{ size_t cap = 0;
  int rc = dx_undexta_size_dev(ctx,DX_FASTA,d_in,n,o->width,&cap);
  if (rc != DX_OK) return rc;
  *d_out = (uint8_t *) dx_device_alloc(ctx,cap + 64);
  if (*d_out == NULL) return DX_E_NOMEM;
  return dx_undexta_dev(ctx,DX_FASTA,d_in,n,o->width,o->upper,*d_out,cap + 64,out_len);
}

static int stream(dx_win *w) { return dx_stream_unpack(w,DX_FASTA); }

int main(int argc, char *argv[])
{ static const dx_tool tool =
    { "undexta", "[-vkU] [-w<int(80)>] ( -i | <path:dexta> ... )", "vkiU", 1, ".dexta", ".fasta",
      { "      -i: source is on standard input.",
        "      -k: do *not* remove the .dexta file on completion.",
        "      -U: use uppercase letters (default is lower case).",
        "      -w: line width for sequence lines.", NULL }, run, stream, 10.0 };
  return dx_cli_main(&tool,argc,argv);
}
