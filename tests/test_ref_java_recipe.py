"""The reference-run recipe (oracle/ref_java): the Processing pre-processor subset is checked on snippets (no JVM is needed
for that): only literal suffixes, colours and conversion calls may change."""
import importlib.util
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
spec = importlib.util.spec_from_file_location("pde2java", ROOT / "oracle" / "ref_java" / "pde2java.py")
pde2java = importlib.util.module_from_spec(spec)
spec.loader.exec_module(pde2java)


def test_literals_colours_and_conversions():
    c = pde2java.convert
    assert c("float a = 0.5*(b+1.)/3;") == "float a = 0.5f*(b+1.f)/3;"
    assert c("x = .125; y = 1e-5; z = 1e-4f; w = 2;") == "x = .125f; y = 1e-5f; z = 1e-4f; w = 2;"
    assert c("a[i][j] = x.r*i + v2.x;") == "a[i][j] = x.r*i + v2.x;"                 # member access is not a literal
    assert c("color bodyColor = #993333; stroke(#000000);") == "int bodyColor = 0xFF993333; stroke(0xFF000000);"
    assert c("img.pixels[k] = color(f);") == "img.pixels[k] = color(f);"              # the FUNCTION color stays
    assert c("t = float(stuff[0]); s /= float(m-2); k = int(x);") == "t = parseFloat(stuff[0]); s /= parseFloat(m-2); k = parseInt(x);"
    assert c("float y = (float)(i-0.5); print(1.5);") == "float y = (float)(i-0.5f); print(1.5f);"   # casts and print( untouched


def test_strings_and_comments_are_left_alone():
    c = pde2java.convert
    src = 'println("dt = 0.5, color #993333"); // scale by 0.5\n/* float(x) 1.0 */ char q = \'.\'; x = 1.0;'
    assert c(src) == 'println("dt = 0.5, color #993333"); // scale by 0.5\n/* float(x) 1.0 */ char q = \'.\'; x = 1.0f;'

