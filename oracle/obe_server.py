"""The reference's TCP front end restated: ``Socket`` (optbayesexpt/obe_socket.py:12-25,88-129) and ``OBE_Server``
(optbayesexpt/obe_server.py:118-315), for the commands tests/test_gpu_server.py sends.

TEST INFRASTRUCTURE.  The wire format is the reference's: a message is its JSON text preceded by the text's length
as 10 zero-padded decimal digits, and every command is one connection (connect, send, receive the reply, close).
Replies are the engine's values as they are (``json.dumps`` of a tuple, a float subclass, or an array's
``tolist()``), as in the reference: nothing is converted on their way.  The server runs whichever engine ``make_obe``
built; with the reference installed (baseline/install_reference.sh) the test drives the reference's own classes
instead.
"""
import json
import socket


class Socket:
    def __init__(self, role, ip_address='127.0.0.1', port=61981):
        self.role = role
        self.ip_address = ip_address
        self.port = port
        self.connection = None
        if role == 'server':
            self.server = socket.socket(socket.AF_INET, socket.SOCK_STREAM)
            self.server.bind((ip_address, port))
            self.server.listen(1)

    def send(self, contents):
        text = json.dumps(contents)
        self.connection.sendall(('%010d' % len(text) + text).encode())

    def _read(self, n):
        data = b''
        while len(data) < n:
            chunk = self.connection.recv(n - len(data))
            if not chunk:
                raise ConnectionError('connection closed inside a message')
            data += chunk
        return data

    def receive(self):
        return json.loads(self._read(int(self._read(10).decode())).decode())

    def tcpcmd(self, command):
        """Client side: one command, one reply."""
        self.connection = socket.socket(socket.AF_INET, socket.SOCK_STREAM)
        try:
            self.connection.connect((self.ip_address, self.port))
            self.send(command)
            return self.receive()
        finally:
            self.connection.close()
            self.connection = None


class OBE_Server(Socket):
    def __init__(self, ip_address='127.0.0.1', port=61981):
        Socket.__init__(self, 'server', ip_address=ip_address, port=port)
        self.obe_engine = None

    def make_obe(self, obe_class, initial_args=(), **kwargs):
        self.obe_engine = obe_class(*initial_args, **kwargs)

    def newdat(self, x, y, s):
        self.obe_engine.pdf_update((x, y, s))

    def _reply(self, message):
        eng, cmd = self.obe_engine, message['command']
        if cmd == 'newdat':
            self.newdat(message['x'], message['y'], message['s'])
            return 'OK'
        if cmd == 'optset':
            return eng.opt_setting()
        if cmd == 'goodset':
            return eng.good_setting(pickiness=message['pickiness'])
        if cmd == 'getmean':
            return eng.mean().tolist()
        if cmd == 'getstd':
            return eng.std().tolist()
        if cmd == 'getcov':
            return eng.covariance().tolist()
        if cmd == 'getset':
            return eng.allsettings.tolist()
        if cmd == 'getcon':
            return eng.cons
        if cmd == 'getpar':
            return eng.parameters.tolist()
        if cmd == 'getwgt':
            return eng.particle_weights.tolist()
        if cmd == 'ready':
            return 'OK'
        raise ValueError(f'unknown command {cmd!r}')

    def run(self):
        """Serve one command per connection until 'done'."""
        while True:
            self.connection, _ = self.server.accept()
            try:
                message = self.receive()
                if message['command'] == 'done':
                    self.send('OK')
                    return
                self.send(self._reply(message))
            finally:
                self.connection.close()
                self.connection = None
